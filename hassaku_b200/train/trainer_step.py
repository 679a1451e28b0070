"""One fused training step of SGDMatrixFactorization (train/trainer.py:133-148 of the reference)."""
import torch

from hassaku_b200 import _C, determinism, nvtx
from hassaku_b200.train.optim import DenseAdam
from hassaku_b200.train.rec_losses import RecommenderSystemLoss


class HostBatchStager:
    """Host batches (the reference loaders) to the device: 3 rotating device staging slots filled on a copy stream, so
    the H2D of batch s+1 overlaps the kernels of batch s.  `stage` returns (slot, u, i); record slot['free'] on the
    compute stream after the batch's last kernel."""

    def __init__(self, device):
        self.device = device
        self._copy_stream = None
        self._slots, self._k = [], 0

    def stage(self, u_host: torch.Tensor, i_host: torch.Tensor):
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        B, N1 = i_host.shape
        if not self._slots or self._slots[0]['i'].shape[1] != N1 or self._slots[0]['i'].shape[0] < B:
            self._slots = [{'u': torch.empty(B, dtype=torch.int64, device=self.device),
                            'i': torch.empty((B, N1), dtype=torch.int64, device=self.device),
                            'ready': torch.cuda.Event(), 'free': torch.cuda.Event()} for _ in range(3)]
            for sl in self._slots:
                sl['free'].record()
        sl = self._slots[self._k % 3]
        self._k += 1
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(sl['free'])
            sl['u'][:B].copy_(u_host.to(torch.int64), non_blocking=True)
            sl['i'][:B].copy_(i_host.to(torch.int64), non_blocking=True)
            sl['ready'].record(self._copy_stream)
        torch.cuda.current_stream().wait_event(sl['ready'])
        return sl, sl['u'][:B], sl['i'][:B]

    def device_batch(self, u_idxs: torch.Tensor, i_idxs: torch.Tensor):
        """(slot or None, u, i): device batches pass through as int64, host batches are staged."""
        if u_idxs.is_cuda and i_idxs.is_cuda:
            return None, u_idxs.to(self.device, torch.int64).contiguous(), i_idxs.to(self.device, torch.int64).contiguous()
        return self.stage(u_idxs, i_idxs)


class FusedMFTrainStep:
    """One training step of SGDMatrixFactorization: trainer.py:133-148 as hsk_mf_train_fused + hsk_adamw_dense."""

    def __init__(self, model, rec_loss: RecommenderSystemLoss, optimizer: DenseAdam):
        if rec_loss.loss_kind not in _C.LOSS_KINDS:
            raise ValueError(f'Loss {rec_loss.name} has no fused kernel')
        self.model, self.rec_loss, self.optimizer = model, rec_loss, optimizer
        self.kind = _C.LOSS_KINDS[rec_loss.loss_kind]
        self.shift = float(rec_loss.neg_shift())
        self.device = model.arena.device
        self.loss_accum = torch.zeros(1, dtype=torch.float64, device=self.device)
        self._stager = HostBatchStager(self.device)

    def __call__(self, u_idxs: torch.Tensor, i_idxs: torch.Tensor, loss_out: torch.Tensor = None):
        """Enqueue one step.  `loss_out` (fp64 [1], device) receives this batch's mean loss added to it; by default
        the epoch accumulator is used."""
        with nvtx.range('hsk.train_step'):
            self._step(u_idxs, i_idxs, loss_out)

    def _step(self, u_idxs, i_idxs, loss_out):
        slot, u, i = self._stager.device_batch(u_idxs, i_idxs)
        loss =self.loss_accum if loss_out is None else loss_out
        if determinism.enabled():
            scratch = determinism.scratch(self, _C.det_scratch_bytes(i.shape[0], i.shape[1], self.model.layout.ld),
                                          self.device)
            _C.mf_train_fused_det(self.model._tables(), self.optimizer.grad_tables, u, i, self.kind, self.shift, loss,
                                  scratch, status=self.model._status())
        else:
            _C.mf_train_fused(self.model._tables(), self.optimizer.grad_tables, u, i, self.kind, self.shift, loss,
                              status=self.model._status())
        if hasattr(self.optimizer, 'mark'):
            self.optimizer.mark(u, i)
        self.optimizer.step_fused()
        if slot is not None:
            slot['free'].record()

    def pop_loss_sum(self) -> float:
        """Host sync: sum of the batch-mean losses since the last call (also surfaces index errors)."""
        v = float(self.loss_accum.item())
        self.loss_accum.zero_()
        self.model.check_status()
        return v
