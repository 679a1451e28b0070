"""torch.use_deterministic_algorithms for hassaku_b200.

The switch is read when work is enqueued, as torch's own ops do.  With it on, every single-GPU train and eval launch that
reduces with floating-point atomics takes its deterministic kernel (hsk_det.cu: fixed summation order, one writer per
row), and work that has no deterministic implementation raises `RuntimeError` (or only warns under `warn_only=True`)."""
import warnings

import torch


def enabled() -> bool:
    """True under `torch.use_deterministic_algorithms(True)` (also with `warn_only=True`)."""
    return torch.are_deterministic_algorithms_enabled()


def alert_not_deterministic(caller: str):
    """torch's contract for an op without a deterministic implementation: raise, or warn under `warn_only=True`."""
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = (f'{caller} does not have a deterministic implementation, but you set '
           "'torch.use_deterministic_algorithms(True)'. You can turn off determinism just for this operation, or you can "
           "use the 'warn_only=True' option, if that's acceptable for your application.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(msg, UserWarning, stacklevel=3)
    else:
        raise RuntimeError(msg)


def scratch(owner, nbytes: int, device) -> torch.Tensor:
    """A device byte buffer of at least `nbytes`, kept on `owner` and grown on demand: the per-step path allocates
    nothing once the batch shape is known (under the switch torch fills every fresh allocation)."""
    buf = owner.__dict__.get('_hsk_det_scratch')
    if buf is None or buf.numel() < nbytes or buf.device != torch.device(device):
        buf = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
        owner.__dict__['_hsk_det_scratch'] = buf
    return buf
