"""ctypes binding of the C-ABI in include/hassaku_b200.h (hassaku_b200/lib/libhassaku_b200.so).

There is NO fallback: if the shared library is missing or a call is made without a CUDA device the error is
raised to the caller.  PyTorch is used only for device memory and streams: every wrapper passes raw device
pointers and the current CUDA stream of the calling thread; ctypes releases the GIL around the call.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('HSK_LIB_PATH') or os.path.join(_HERE, 'lib', 'libhassaku_b200.so')   # override: experimental builds

LOSS_KINDS = {'bpr': 0, 'sampled_softmax': 1, 'bce': 2}
STATUS_BAD_INDEX = 1
STATUS_CAPACITY = 2
STATUS_SAMPLER_ROUNDS = 4
STATUS_BARRIER_TIMEOUT = 8
PRECISIONS = {'fp32': 0, 'tf32': 1, 'bf16': 2}
TRAIN_VARIANTS = {'auto': 0, 'regs': 1, 'ring': 2, 'q': 3}   # HSK_TRAIN_* of hsk_mf_train_fused_v
# kernel choice used by mf_train_fused / mf_train_fused_n of THIS binding (parity tests and scripts/kbench.py set it; the
# library itself holds no state: the variant is an argument of hsk_mf_train_fused_v)
TRAIN_VARIANT = 'auto'
EVAL_TC_VARIANTS = {'auto': 0, 'single': 1, 'pair': 2}      # HSK_EVAL_TC_* of hsk_eval_topk_tc_v
EVAL_TC_VARIANT = 'auto'


class HskError(RuntimeError):
    pass


class MfTables(C.Structure):
    """struct hsk_mf_tables (include/hassaku_b200.h)."""
    _fields_ = [('Uw', C.c_void_p), ('Vw', C.c_void_p), ('Ub', C.c_void_p), ('Ib', C.c_void_p), ('Gb', C.c_void_p),
                ('n_users', C.c_int64), ('n_items', C.c_int64), ('d', C.c_int32), ('ld', C.c_int32)]


class RowSegment(C.Structure):
    """struct hsk_row_segment (include/hassaku_b200.h)."""
    _fields_ = [('offset', C.c_int64), ('n_rows', C.c_int64), ('ld', C.c_int32), ('stamps', C.c_void_p)]


MAX_PEERS = 8
PEER_HANDLE_BYTES = 64


class PeerItems(C.Structure):
    """struct hsk_peer_items (include/hassaku_b200.h): the item side of every rank's tables, mapped into this process."""
    _fields_ = [('world', C.c_int32), ('V', C.c_void_p * MAX_PEERS), ('gV', C.c_void_p * MAX_PEERS),
                ('Ib', C.c_void_p * MAX_PEERS), ('gIb', C.c_void_p * MAX_PEERS), ('stamps', C.c_void_p * MAX_PEERS)]


class PeerFlags(C.Structure):
    """struct hsk_peer_flags: every rank's barrier flag array (hsk_peer_barrier)."""
    _fields_ = [('world', C.c_int32), ('rank', C.c_int32), ('flags', C.c_void_p * MAX_PEERS)]


_lib = None


def _declare(lib):
    vp, i32, i64, f32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
    T = C.POINTER(MfTables)
    sig = {
        'hsk_last_error': (C.c_char_p, []),
        'hsk_version': (i32, []),
        'hsk_device_info': (i32, [C.POINTER(C.c_int)] * 3 + [C.POINTER(C.c_int64)] * 2),
        'hsk_mf_scores': (i32, [T, vp, vp, i32, i32, vp, vp, vp]),
        'hsk_rec_loss': (i32, [vp, vp, i32, i32, i32, f32, f32, vp, vp, vp, vp]),
        'hsk_mf_scatter_grads': (i32, [T, T, vp, vp, vp, i32, i32, vp, vp]),
        'hsk_mf_train_fused': (i32, [T, T, vp, vp, i32, i32, i32, f32, vp, vp, vp, vp, vp]),
        'hsk_mf_train_fused_n': (i32, [T, T, vp, vp, i32, i32, i64, i32, f32, vp, vp, vp, vp, vp]),
        'hsk_mf_train_fused_v': (i32, [T, T, vp, vp, i32, i32, i64, i32, f32, vp, vp, vp, vp, i32, vp]),
        'hsk_eval_topk_tc_shards_scratch_bytes': (i64, [i32, vp, i32, i32]),
        'hsk_eval_topk_tc_shards': (i32, [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, i32, i64, vp, vp, i32, vp, vp, vp, i64, vp, vp]),
        'hsk_rescore_topk_shards': (i32, [T, vp, vp, vp, i32, vp, i32, vp, vp, i32, i32, vp, vp, vp, vp]),
        'hsk_topk_tag_means': (i32, [vp, i32, i32, vp, i64, i32, C.POINTER(C.c_int), i32, vp, vp, vp]),
        'hsk_peer_export': (i32, [vp, vp, C.POINTER(C.c_int64)]),
        'hsk_peer_open': (i32, [vp, C.POINTER(C.c_void_p)]),
        'hsk_peer_close': (i32, [vp]),
        'hsk_peer_barrier': (i32, [C.POINTER(PeerFlags), vp, vp, vp]),
        'hsk_mf_train_fused_peer': (i32, [T, T, C.POINTER(PeerItems), vp, vp, i32, i32, i64, i32, f32, vp, i64, vp, vp, vp]),
        'hsk_gather_rows': (i32, [vp, i32, vp, i64, i64, vp, vp, vp]),
        'hsk_shard_local_index': (i32, [vp, i64, i32, i64, vp, vp]),
        'hsk_scatter_add_rows': (i32, [vp, i32, vp, i64, i64, vp, vp, vp]),
        'hsk_row_stamp': (i32, [i64]),
        'hsk_mark_rows': (i32, [vp, i64, i64, vp, i64, vp, vp]),
        'hsk_mark_batch': (i32, [vp, vp, i32, i32, i64, i64, vp, vp, i64, vp, vp]),
        'hsk_adamw_dense_rows': (i32, [vp, vp, vp, vp, i64, C.POINTER(RowSegment), i32, f64, f64, f64, f64, f64, i64, vp, vp, i32, i32, vp]),
        'hsk_adamw_dense_rows_lag': (i32, [vp, vp, vp, vp, i64, C.POINTER(RowSegment), i32, C.POINTER(vp), C.POINTER(vp), i32,
                                           f64, f64, f64, f64, f64, i64, i32, i32, vp]),
        'hsk_adamw_lag_sync': (i32, [vp, vp, i64, C.POINTER(RowSegment), i32, C.POINTER(vp), C.POINTER(vp), f64, f64, i64, i32,
                                     vp]),
        'hsk_rescore_topk': (i32, [T, vp, i32, i64, i64, vp, vp, i32, i32, vp, vp, vp, vp]),
        'hsk_rescore_scores': (i32, [T, vp, i32, i64, i64, vp, i32, vp, vp, vp]),
        'hsk_topk_combine': (i32, [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp]),
        'hsk_shard_block_rows': (i64, [i32, i32]),
        'hsk_route_scratch_bytes': (i64, [i64, i32]),
        'hsk_route_items': (i32, [vp, i64, i64, i32, i32, i32, vp, vp, vp, vp, i64, vp, vp]),
        'hsk_shard_pack': (i32, [vp, vp, i32, i64, vp, i32, i32, vp, vp, vp]),
        'hsk_shard_unpack_add': (i32, [vp, i32, i64, vp, i32, i32, vp, vp, vp, i64, vp, vp, vp]),
        'hsk_shard_unpack_ordered': (i32, [vp, i32, i64, vp, i32, i32, vp, vp, vp, i64, vp, vp, vp]),
        'hsk_adamw_dense': (i32, [vp, vp, vp, vp, i64, f64, f64, f64, f64, f64, i64, i32, i32, i32, vp]),
        'hsk_sample_negatives': (i32, [vp, vp, i32, i32, i64, i64, vp, vp, C.c_uint64, C.c_uint64, i32, vp, vp, vp, vp]),
        'hsk_adagrad_dense': (i32, [vp, vp, vp, i64, f64, f64, f64, i32, vp]),
        'hsk_mark_touched': (i32, [vp, vp, i32, i32, i64, i64, vp, vp, vp]),
        'hsk_adamw_rows_lazy': (i32, [vp, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, f64, f64, f64, f64, f64, i64, vp]),
        'hsk_adamw_consts': (i32, [f64, f64, f64, f64, f64, i64, vp]),
        'hsk_adamw_dense_graph': (i32, [vp, vp, vp, vp, i64, vp, i32, i32, i32, vp]),
        'hsk_eval_topk_scratch_bytes': (i64, [i32, i64, i32]),
        'hsk_eval_topk': (i32, [T, vp, vp, i64, i32, i64, i64, vp, vp, i32, vp, vp, vp, i64, vp, vp]),
        'hsk_eval_tc_kpad': (i32, [i32, i32]),
        'hsk_pack_rows': (i32, [vp, i32, i32, vp, i64, i64, vp, i32, i32, vp, vp]),
        'hsk_eval_topk_tc_scratch_bytes': (i64, [i32, i64, i32]),
        'hsk_eval_topk_tc': (i32, [vp, vp, i32, i32, vp, vp, vp, vp, vp, i32, i64, i64, i64, i64, vp, vp, i32, vp, vp, vp,
                                   i64, vp, vp]),
        'hsk_eval_topk_tc_v': (i32, [vp, vp, i32, i32, vp, vp, vp, vp, vp, i32, i64, i64, i64, i64, vp, vp, i32, vp, vp, vp,
                                     i64, vp, i32, vp]),
        'hsk_topk_merge': (i32, [vp, vp, i32, i32, i32, vp, vp, vp]),
        'hsk_topk_dense': (i32, [vp, i32, i64, i64, i32, vp, vp, vp]),
        'hsk_rank_metrics': (i32, [vp, i32, i32, C.POINTER(C.c_int), i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]),
        'hsk_rank_metrics_dense': (i32, [vp, i32, i32, C.POINTER(C.c_int), i32, vp, vp, i64, vp, i32, vp, vp, vp, vp,
                                         vp]),
        'hsk_det_scratch_bytes': (i64, [i32, i32, i32]),
        'hsk_mf_scatter_grads_det': (i32, [T, T, vp, vp, vp, i32, i32, vp, i64, vp, vp]),
        'hsk_mf_train_fused_det': (i32, [T, T, vp, vp, i32, i32, i32, f32, vp, vp, vp, vp, i64, vp, vp]),
        'hsk_mf_train_fused_det_n': (i32, [T, T, vp, vp, i32, i32, i64, i32, f32, vp, vp, vp, vp, i64, vp, vp]),
        'hsk_rec_loss_det': (i32, [vp, vp, i32, i32, i32, f32, f32, vp, vp, vp, vp, i64, vp]),
        'hsk_rank_metrics_sums_det': (i32, [vp, i32, i32, vp, vp, i32, vp, vp]),
        'hsk_mf_train_fused_pack': (i32, [T, T, i64, i32, vp, i32, vp, vp, i32, i32, i32, f32, vp, vp, vp]),
        'hsk_adamw_pack': (i32, [vp, vp, vp, vp, i64, i32, vp, i32, vp, C.POINTER(RowSegment), i32, i64, i32, vp, vp]),
        'hsk_adamw_consts_table': (i32, [vp, vp, i32, f64, f64, f64, i64, i32, vp]),
        'hsk_eval_topk_pack_scratch_bytes': (i64, [i32, i64, i32, i32]),
        'hsk_eval_topk_pack': (i32, [T, i64, i32, vp, i32, vp, i32, vp, vp, i32, vp, vp, vp, i64, vp, vp]),
        'hsk_rank_metrics_pack': (i32, [vp, i32, i32, C.POINTER(C.c_int), i32, vp, vp, vp, vp, i32, vp, i32, vp, i32, vp, vp, vp,
                                        vp, vp]),
        'hsk_rank_metrics_sums_det_pack': (i32, [vp, i32, i32, i32, vp, vp, i32, i32, vp, i32, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return sig


def lib():
    """Load the shared library (once).  Raises HskError with build instructions if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HskError(f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                           f'or `make -C hassaku_b200/csrc` (nvcc, sm_100a). There is no CPU fallback.')
        l = C.CDLL(LIB_PATH)
        _declare(l)
        _lib = l
    return _lib


def exported_symbols():
    return list(_declare(lib()).keys())


def _check(rc: int, who: str):
    if rc != 0:
        raise HskError(f'{who} failed ({rc}): {lib().hsk_last_error().decode()}')


class _on_device_of:
    """Device guard of one launch: every CUDA tensor argument must live on ONE device; the launch goes to that device's
    current stream with that device current (the library launches on the calling thread's current device), whatever
    device the caller had selected (a model on cuda:1 while cuda:0 is current)."""
    __slots__ = ('dev', 'prev')

    def __init__(self, *tensors):
        dev = None
        for t in tensors:
            if t is None or not isinstance(t, torch.Tensor) or not t.is_cuda:
                continue
            if dev is None:
                dev = t.device
            elif t.device != dev:
                raise HskError(f'tensors of one call live on different devices ({dev} and {t.device})')
        self.dev, self.prev = dev, None

    def __enter__(self) -> int:
        if self.dev is None:
            return torch.cuda.current_stream().cuda_stream
        if torch.cuda.current_device() != self.dev.index:
            self.prev = torch.cuda.current_device()
            torch.cuda.set_device(self.dev)
        return torch.cuda.current_stream(self.dev).cuda_stream

    def __exit__(self, *exc):
        if self.prev is not None:
            torch.cuda.set_device(self.prev)
        return False


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str, contiguous: bool = True):
    if not t.is_cuda:
        raise HskError(f'{name} must be a CUDA tensor: hassaku_b200 has no CPU path')
    if t.dtype != dtype:
        raise HskError(f'{name} must be {dtype}, got {t.dtype}')
    if contiguous and not t.is_contiguous():
        raise HskError(f'{name} must be contiguous')
    return t


def make_tables(Uw, Vw, Ub, Ib, Gb, d: int) -> MfTables:
    """Uw/Vw: [rows, ld] fp32 CUDA with stride (ld, 1) (may be a [:, :d] view of padded storage)."""
    for n, w in (('Uw', Uw), ('Vw', Vw)):
        if not w.is_cuda or w.dtype != torch.float32 or w.dim() != 2 or w.stride(1) != 1:
            raise HskError(f'{n} must be a 2-D fp32 CUDA tensor with unit inner stride (no CPU path)')
    if Uw.stride(0) != Vw.stride(0):
        raise HskError('Uw and Vw must share one leading dimension')
    return MfTables(Uw.data_ptr(), Vw.data_ptr(), _ptr(Ub), _ptr(Ib), _ptr(Gb), Uw.shape[0], Vw.shape[0], d,
                    Uw.stride(0))


def device_info():
    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    l2, hbm = C.c_int64(), C.c_int64()
    _check(lib().hsk_device_info(C.byref(sm), C.byref(ma), C.byref(mi), C.byref(l2), C.byref(hbm)), 'hsk_device_info')
    return {'sm_count': sm.value, 'cc': (ma.value, mi.value), 'l2_bytes': l2.value, 'hbm_bytes': hbm.value}


def mf_scores(tables: MfTables, u_idx, i_idx, scores, status=None):
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(scores, torch.float32, 'scores')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, scores, status) as st:
        _check(lib().hsk_mf_scores(C.byref(tables), u_idx.data_ptr(), i_idx.data_ptr(), B, N1, scores.data_ptr(),
                                   _ptr(status), st), 'hsk_mf_scores')


def rec_loss(scores, labels, loss_kind: int, neg_shift: float, grad_scale: float, loss_accum, dscores=None,
             shifted_out=None):
    _req(scores, torch.float32, 'scores'); _req(loss_accum, torch.float64, 'loss_accum')
    if labels is not None:
        _req(labels, torch.float64, 'labels')
    B, N1 = scores.shape
    with _on_device_of(scores, labels, loss_accum, dscores, shifted_out) as st:
        _check(lib().hsk_rec_loss(scores.data_ptr(), _ptr(labels), B, N1, loss_kind, neg_shift, grad_scale,
                                  loss_accum.data_ptr(), _ptr(dscores), _ptr(shifted_out), st), 'hsk_rec_loss')


def mf_scatter_grads(tables: MfTables, grads: MfTables, u_idx, i_idx, dscores, status=None):
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(dscores, torch.float32, 'dscores')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, dscores, status) as st:
        _check(lib().hsk_mf_scatter_grads(C.byref(tables), C.byref(grads), u_idx.data_ptr(), i_idx.data_ptr(),
                                          dscores.data_ptr(), B, N1, _ptr(status), st), 'hsk_mf_scatter_grads')


def mf_train_fused(tables: MfTables, grads: MfTables, u_idx, i_idx, loss_kind: int, neg_shift: float, loss_accum,
                   scores_out=None, dscores_out=None, status=None, B_global: Optional[int] = None, variant: Optional[str] = None):
    """hsk_mf_train_fused_v: B_global (default: the batch itself) keeps the normalisers global in the sharded step;
    variant (default: module-level TRAIN_VARIANT) selects the kernel."""
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(loss_accum, torch.float64, 'loss_accum')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, loss_accum, scores_out, dscores_out, status) as st:
        _check(lib().hsk_mf_train_fused_v(C.byref(tables), C.byref(grads), u_idx.data_ptr(), i_idx.data_ptr(), B, N1,
                                          B if B_global is None else B_global, loss_kind, neg_shift, loss_accum.data_ptr(),
                                          _ptr(scores_out), _ptr(dscores_out), _ptr(status),
                                          TRAIN_VARIANTS[variant or TRAIN_VARIANT], st), 'hsk_mf_train_fused')


def mf_train_fused_n(tables: MfTables, grads: MfTables, u_idx, i_idx, B_global: int, loss_kind: int, neg_shift: float,
                     loss_accum, status=None):
    mf_train_fused(tables, grads, u_idx, i_idx, loss_kind, neg_shift, loss_accum, status=status, B_global=B_global)


def peer_export(t: torch.Tensor):
    """(handle bytes, offset) of the device allocation behind `t` for the peers of this node (hsk_peer_export)."""
    h = C.create_string_buffer(PEER_HANDLE_BYTES)
    off = C.c_int64(0)
    with _on_device_of(t):
        _check(lib().hsk_peer_export(t.data_ptr(), h, C.byref(off)), 'hsk_peer_export')
    return bytes(h.raw), int(off.value)


def peer_open(handle: bytes, device) -> int:
    """Map a peer's allocation into this process; returns its base address here (hsk_peer_open)."""
    base = C.c_void_p(0)
    with torch.cuda.device(device):
        _check(lib().hsk_peer_open(C.create_string_buffer(handle, PEER_HANDLE_BYTES), C.byref(base)), 'hsk_peer_open')
    return int(base.value)


def peer_close(base: int):
    _check(lib().hsk_peer_close(C.c_void_p(base)), 'hsk_peer_close')


def make_peer_items(V_ptrs, gV_ptrs, Ib_ptrs=None, gIb_ptrs=None, stamp_ptrs=None) -> PeerItems:
    """Device addresses (ints, valid in THIS process) of every rank's local item tables, rank order."""
    G = len(V_ptrs)
    if not 1 <= G <= MAX_PEERS:
        raise ValueError(f'peer exchange supports 1..{MAX_PEERS} ranks, got {G}')
    p = PeerItems()
    p.world = G
    for q in range(G):
        p.V[q], p.gV[q] = V_ptrs[q], gV_ptrs[q]
        p.Ib[q] = Ib_ptrs[q] if Ib_ptrs else None
        p.gIb[q] = gIb_ptrs[q] if gIb_ptrs else None
        p.stamps[q] = stamp_ptrs[q] if stamp_ptrs else None
    return p


def make_peer_flags(flag_ptrs, rank: int) -> PeerFlags:
    f = PeerFlags()
    f.world, f.rank = len(flag_ptrs), rank
    for q, a in enumerate(flag_ptrs):
        f.flags[q] = a
    return f


def peer_barrier(flags: PeerFlags, epoch, status=None):
    """hsk_peer_barrier on the current stream of epoch's device."""
    _req(epoch, torch.int32, 'epoch')
    with _on_device_of(epoch, status) as st:
        _check(lib().hsk_peer_barrier(C.byref(flags), epoch.data_ptr(), _ptr(status), st), 'hsk_peer_barrier')


def mf_train_fused_peer(tables: MfTables, grads: MfTables, peers: PeerItems, u_idx, i_idx, B_global: int, loss_kind: int,
                        neg_shift: float, loss_accum, step: int = 0, step_dev=None, status=None):
    """hsk_mf_train_fused_peer: the step kernel over peer-mapped item shards (rows <= 128 floats)."""
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(loss_accum, torch.float64, 'loss_accum')
    if step_dev is not None:
        _req(step_dev, torch.int64, 'step_dev')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, loss_accum, step_dev, status) as st:
        _check(lib().hsk_mf_train_fused_peer(C.byref(tables), C.byref(grads), C.byref(peers), u_idx.data_ptr(), i_idx.data_ptr(),
                                             B, N1, B_global, loss_kind, neg_shift, loss_accum.data_ptr(), step, _ptr(step_dev),
                                             _ptr(status), st), 'hsk_mf_train_fused_peer')


def gather_rows(src, idx, dst, status=None):
    """dst[r, :] = src[idx[r], :]; src/dst 2-D fp32 with the same (padded) leading dimension."""
    _req(idx, torch.int64, 'idx')
    with _on_device_of(src, idx, dst, status) as st:
        _check(lib().hsk_gather_rows(src.data_ptr(), src.stride(0), idx.data_ptr(), idx.numel(), src.shape[0],
                                     dst.data_ptr(), _ptr(status), st), 'hsk_gather_rows')


def shard_local_index(idx, world: int, rank_stride: int, out=None):
    """out = (idx % world) * rank_stride + idx // world (owner-sharded row numbering, hassaku_b200/sharded.py)."""
    _req(idx, torch.int64, 'idx')
    if out is None:
        out = torch.empty_like(idx)
    with _on_device_of(idx, out) as st:
        _check(lib().hsk_shard_local_index(idx.data_ptr(), idx.numel(), world, rank_stride, out.data_ptr(), st),
               'hsk_shard_local_index')
    return out


def scatter_add_rows(dst, idx, src, status=None):
    """dst[idx[r], :] += src[r, :]."""
    _req(idx, torch.int64, 'idx')
    with _on_device_of(dst, idx, src, status) as st:
        _check(lib().hsk_scatter_add_rows(dst.data_ptr(), dst.stride(0), idx.data_ptr(), idx.numel(), dst.shape[0],
                                          src.data_ptr(), _ptr(status), st), 'hsk_scatter_add_rows')


# ---- device-side routing of the item-sharded step (hsk_shard.cu) ----
def shard_block_rows(capq: int, ld: int) -> int:
    return int(lib().hsk_shard_block_rows(capq, ld))


def route_scratch_bytes(n_items: int, world: int) -> int:
    return int(lib().hsk_route_scratch_bytes(n_items, world))


def route_items(i_idx, n_items: int, world: int, capq: int, ld: int, req_rows, req_count, compact_idx, scratch, status=None):
    """Distinct item ids of the batch grouped by owner -> req_rows [world, capq] int32 (-1 padded), req_count [world],
    compact_idx (int64, shape of i_idx): row of each slot in the compact table [world * block_rows, ld]."""
    _req(i_idx, torch.int64, 'i_idx'); _req(req_rows, torch.int32, 'req_rows'); _req(req_count, torch.int32, 'req_count')
    _req(compact_idx, torch.int64, 'compact_idx'); _req(scratch, torch.uint8, 'scratch')
    if req_rows.numel() != world * capq or req_count.numel() != world or compact_idx.numel() != i_idx.numel():
        raise HskError('route_items: req_rows must be [world, capq], req_count [world], compact_idx like i_idx')
    with _on_device_of(i_idx, req_rows, req_count, compact_idx, scratch, status) as st:
        _check(lib().hsk_route_items(i_idx.data_ptr(), i_idx.numel(), n_items, world, capq, ld, req_rows.data_ptr(),
                                     req_count.data_ptr(), compact_idx.data_ptr(), scratch.data_ptr(), scratch.numel(),
                                     _ptr(status), st), 'hsk_route_items')


def shard_pack(V2d, Ib, rows, world: int, capq: int, out, status=None):
    """rows [world, capq] int32 (local rows the peers want, -1 = padding) -> out [world, block_rows, ld] send blocks."""
    _req(rows, torch.int32, 'rows'); _req(out, torch.float32, 'out')
    ld = V2d.stride(0)
    if out.numel() != world * shard_block_rows(capq, ld) * ld:
        raise HskError('shard_pack: out must hold world * block_rows * ld floats')
    with _on_device_of(V2d, Ib, rows, out, status) as st:
        _check(lib().hsk_shard_pack(V2d.data_ptr(), _ptr(Ib), ld, V2d.shape[0], rows.data_ptr(), world, capq, out.data_ptr(),
                                    _ptr(status), st), 'hsk_shard_pack')


def shard_unpack_add(inp, rows, world: int, capq: int, gV2d, gIb=None, stamps=None, step: int = 0, step_dev=None, status=None,
                     ordered: bool = False):
    """Owner side of the sparse exchange: the peers' row / bias gradients into gV2d / gIb, rows stamped.  `ordered`:
    hsk_shard_unpack_ordered (every row composed in increasing rank order and stored, no atomics) instead of
    hsk_shard_unpack_add."""
    _req(rows, torch.int32, 'rows'); _req(inp, torch.float32, 'inp')
    ld = gV2d.stride(0)
    if stamps is not None:
        _req(stamps, torch.uint8, 'stamps')
    if step_dev is not None:
        _req(step_dev, torch.int64, 'step_dev')
    name = 'hsk_shard_unpack_ordered' if ordered else 'hsk_shard_unpack_add'
    with _on_device_of(inp, rows, gV2d, gIb, stamps, step_dev, status) as st:
        _check(getattr(lib(), name)(inp.data_ptr(), ld, gV2d.shape[0], rows.data_ptr(), world, capq, gV2d.data_ptr(),
                                    _ptr(gIb), _ptr(stamps), step, _ptr(step_dev), _ptr(status), st), name)


def adamw_dense(p, m, v, g, lr, beta1, beta2, eps, weight_decay, step: int, arith: int = 0, adam_l2: bool = False,
                zero_grad: bool = True):
    for n, t in (('p', p), ('m', m), ('v', v), ('g', g)):
        _req(t, torch.float32, n)
    n = p.numel()
    if not (m.numel() == n and v.numel() == n and g.numel() == n):
        raise HskError('adamw_dense: p, m, v, g must have the same number of elements')
    with _on_device_of(p, m, v, g) as st:
        _check(lib().hsk_adamw_dense(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), n, lr, beta1, beta2, eps,
                                     weight_decay, step, arith, int(adam_l2), int(zero_grad), st), 'hsk_adamw_dense')


def row_stamp(step: int) -> int:
    return int(lib().hsk_row_stamp(step))


def mark_rows(idx, n_rows: int, stamps, step: int = 0, step_dev=None):
    _req(idx, torch.int64, 'idx'); _req(stamps, torch.uint8, 'stamps')
    if step_dev is not None:
        _req(step_dev, torch.int64, 'step_dev')
    with _on_device_of(idx, stamps, step_dev) as st:
        _check(lib().hsk_mark_rows(idx.data_ptr(), idx.numel(), n_rows, stamps.data_ptr(), step, _ptr(step_dev), st),
               'hsk_mark_rows')


def mark_batch(u_idx, i_idx, n_users: int, n_items: int, stamps_users, stamps_items, step: int = 0, step_dev=None):
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx')
    for n, t in (('stamps_users', stamps_users), ('stamps_items', stamps_items)):
        if t is not None:
            _req(t, torch.uint8, n)
    if step_dev is not None:
        _req(step_dev, torch.int64, 'step_dev')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, stamps_users, stamps_items, step_dev) as st:
        _check(lib().hsk_mark_batch(u_idx.data_ptr(), i_idx.data_ptr(), B, N1, n_users, n_items, _ptr(stamps_users),
                                    _ptr(stamps_items), step, _ptr(step_dev), st), 'hsk_mark_batch')


def adamw_dense_rows(p, m, v, g, segments, lr, beta1, beta2, eps, weight_decay, step: int, arith: int = 0,
                     adam_l2: bool = False, consts_dev=None, step_dev=None):
    """segments: iterable of (offset, n_rows, ld, stamps uint8 tensor) — the row-structured parts of the arena whose
    gradient traffic is skipped for rows not stamped this step; everything else takes the plain dense path."""
    for n, t in (('p', p), ('m', m), ('v', v), ('g', g)):
        _req(t, torch.float32, n)
    segs, arr = _row_segments(segments, 'adamw_dense_rows')
    if consts_dev is not None:
        _req(consts_dev, torch.float32, 'consts_dev'); _req(step_dev, torch.int64, 'step_dev')
    with _on_device_of(p, m, v, g, consts_dev, step_dev, *[sg[3] for sg in segs]) as st:
        _check(lib().hsk_adamw_dense_rows(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), p.numel(), arr, len(segs),
                                          lr, beta1, beta2, eps, weight_decay, step, _ptr(consts_dev), _ptr(step_dev), arith,
                                          int(adam_l2), st), 'hsk_adamw_dense_rows')


def adamw_dense_rows_lag(p, m, v, g, segments, bases, lag: int, lr, beta1, beta2, eps, weight_decay, step: int,
                         arith: int = 0, adam_l2: bool = False):
    """adamw_dense_rows with the segments' m and v written back once every `lag` steps (hsk_adamw_dense_rows_lag).
    bases: per segment (base_in, base_out), two [n_rows] uint8 tensors; swap them after the call."""
    for n, t in (('p', p), ('m', m), ('v', v), ('g', g)):
        _req(t, torch.float32, n)
    segs, arr = _row_segments(segments, 'adamw_dense_rows_lag')
    b_in, b_out = _lag_bases(segs, bases, 'adamw_dense_rows_lag')
    with _on_device_of(p, m, v, g, *[sg[3] for sg in segs], *[b for pair in bases for b in pair]) as st:
        _check(lib().hsk_adamw_dense_rows_lag(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), p.numel(), arr,
                                              len(segs), b_in, b_out, lag, lr, beta1, beta2, eps, weight_decay, step, arith,
                                              int(adam_l2), st), 'hsk_adamw_dense_rows_lag')


def adamw_lag_sync(m, v, segments, bases, beta1, beta2, step: int, arith: int = 0):
    """every row of the segments to step `step` (hsk_adamw_lag_sync); swap the bases after the call"""
    for n, t in (('m', m), ('v', v)):
        _req(t, torch.float32, n)
    if m.numel() != v.numel():
        raise HskError('adamw_lag_sync: m and v must have the same number of elements')
    segs, arr = _row_segments(segments, 'adamw_lag_sync')
    b_in, b_out = _lag_bases(segs, bases, 'adamw_lag_sync')
    with _on_device_of(m, v, *[b for pair in bases for b in pair]) as st:
        _check(lib().hsk_adamw_lag_sync(m.data_ptr(), v.data_ptr(), m.numel(), arr, len(segs), b_in, b_out, beta1, beta2,
                                        step, arith, st), 'hsk_adamw_lag_sync')


def _lag_bases(segs, bases, who):
    bases = list(bases)
    if len(bases) != len(segs):
        raise HskError(f'{who}: one (base_in, base_out) pair per segment')
    b_in, b_out = (C.c_void_p * max(len(segs), 1))(), (C.c_void_p * max(len(segs), 1))()
    for k, ((_off, rows, _ld, _st), (bi, bo)) in enumerate(zip(segs, bases)):
        _req(bi, torch.uint8, 'base_in'); _req(bo, torch.uint8, 'base_out')
        if bi.numel() < rows or bo.numel() < rows:
            raise HskError(f'{who}: base array shorter than the segment')
        b_in[k], b_out[k] = bi.data_ptr(), bo.data_ptr()
    return b_in, b_out


def _row_segments(segments, who):
    segs = list(segments)
    arr = (RowSegment * max(len(segs), 1))()
    for k, (off, rows, ld, stamps) in enumerate(segs):
        _req(stamps, torch.uint8, 'stamps')
        if stamps.numel() < rows:
            raise HskError(f'{who}: stamp array shorter than the segment')
        arr[k] = RowSegment(off, rows, ld, stamps.data_ptr())
    return segs, arr


# ---- trial pack: M models of one shape, [M, stride] arenas ----
def _pack_rows(name, t, n_trials: int):
    """t: [n_trials, stride] fp32 CUDA, rows contiguous -> stride."""
    _req(t, torch.float32, name)
    if t.dim() != 2 or t.shape[0] != n_trials:
        raise HskError(f'{name} must be [n_trials, stride] with n_trials = {n_trials}')
    return t.shape[1]


def mf_train_fused_pack(tables: MfTables, grads: MfTables, trial_stride: int, n_trials: int, active, u_idx, i_idx,
                        loss_kind: int, neg_shift: float, loss_accum, status=None):
    """hsk_mf_train_fused_pack: the fused step of every trial listed in `active` (int32 device) on one shared batch;
    tables / grads = trial 0's, trial j's at + j * trial_stride elements; loss_accum fp64 [n_trials]."""
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(active, torch.int32, 'active')
    _req(loss_accum, torch.float64, 'loss_accum')
    if loss_accum.numel() != n_trials:
        raise HskError(f'loss_accum must hold n_trials = {n_trials} accumulators')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, active, loss_accum, status) as st:
        _check(lib().hsk_mf_train_fused_pack(C.byref(tables), C.byref(grads), trial_stride, n_trials, active.data_ptr(),
                                             active.numel(), u_idx.data_ptr(), i_idx.data_ptr(), B, N1, loss_kind, neg_shift,
                                             loss_accum.data_ptr(), _ptr(status), st), 'hsk_mf_train_fused_pack')


def adamw_pack(p, m, v, g, active, consts_dev, segments=(), step: int = 0, adam_l2: bool = False, status=None):
    """hsk_adamw_pack over [n_trials, stride] arenas: consts_dev fp32 [n_trials, 8] (this step's hsk_adamw_consts per
    trial); segments (offset inside one trial's row, n_rows, ld, stamps) select the row-stamped form."""
    n_trials = p.shape[0]
    stride = _pack_rows('p', p, n_trials)
    for n, t in (('m', m), ('v', v), ('g', g)):
        if _pack_rows(n, t, n_trials) != stride:
            raise HskError('adamw_pack: p, m, v, g must have one shape')
    _req(active, torch.int32, 'active'); _req(consts_dev, torch.float32, 'consts_dev')
    if consts_dev.numel() != 8 * n_trials:
        raise HskError(f'consts_dev must be [n_trials, 8] = [{n_trials}, 8]')
    segs, arr = _row_segments(segments, 'adamw_pack')
    with _on_device_of(p, m, v, g, active, consts_dev, status, *[sg[3] for sg in segs]) as st:
        _check(lib().hsk_adamw_pack(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), stride, n_trials, active.data_ptr(),
                                    active.numel(), consts_dev.data_ptr(), arr, len(segs), step, int(adam_l2), _ptr(status), st),
               'hsk_adamw_pack')


def adamw_consts_table(lrs, wds, beta1: float, beta2: float, eps: float, first_step: int, n_steps: int, out_host=None):
    """Host fp32 [n_steps, n_trials, 8]: hsk_adamw_consts of trial j at step first_step + s (hsk_adamw_consts_table)."""
    M = len(lrs)
    if len(wds) != M:
        raise HskError('adamw_consts_table: one weight decay per learning rate')
    if out_host is None:
        out_host = torch.empty((n_steps, M, 8), dtype=torch.float32)
    if out_host.is_cuda or out_host.dtype != torch.float32 or out_host.numel() < n_steps * M * 8 or not out_host.is_contiguous():
        raise HskError('adamw_consts_table: out_host must be a contiguous host fp32 tensor of n_steps * n_trials * 8')
    lr_a = (C.c_double * M)(*[float(x) for x in lrs])
    wd_a = (C.c_double * M)(*[float(x) for x in wds])
    _check(lib().hsk_adamw_consts_table(lr_a, wd_a, M, beta1, beta2, eps, first_step, n_steps, out_host.data_ptr()),
           'hsk_adamw_consts_table')
    return out_host


def adagrad_dense(p, state_sum, g, lr, eps=1e-10, weight_decay=0.0, zero_grad=True):
    for n, t in (('p', p), ('state_sum', state_sum), ('g', g)):
        _req(t, torch.float32, n)
    with _on_device_of(p, state_sum, g) as st:
        _check(lib().hsk_adagrad_dense(p.data_ptr(), state_sum.data_ptr(), g.data_ptr(), p.numel(), lr, eps, weight_decay,
                                       int(zero_grad), st), 'hsk_adagrad_dense')


def mark_touched(u_idx, i_idx, n_users: int, n_items: int, touched_users, touched_items):
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx')
    _req(touched_users, torch.uint8, 'touched_users'); _req(touched_items, torch.uint8, 'touched_items')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, touched_users, touched_items) as st:
        _check(lib().hsk_mark_touched(u_idx.data_ptr(), i_idx.data_ptr(), B, N1, n_users, n_items, touched_users.data_ptr(),
                                      touched_items.data_ptr(), st), 'hsk_mark_touched')


def adamw_rows_lazy(p2d, m2d, v2d, g2d, touched, lr, beta1, beta2, eps, weight_decay, step: int, bias=None):
    """p2d/m2d/v2d/g2d: [rows, ld] fp32 views with the same padded leading dimension; bias: optional (p, m, v, g) vectors."""
    _req(touched, torch.uint8, 'touched')
    pb, mb, vb, gb = bias if bias is not None else (None, None, None, None)
    with _on_device_of(p2d, m2d, v2d, g2d, touched, pb) as st:
        _check(lib().hsk_adamw_rows_lazy(p2d.data_ptr(), m2d.data_ptr(), v2d.data_ptr(), g2d.data_ptr(), p2d.shape[0],
                                         p2d.stride(0), _ptr(pb), _ptr(mb), _ptr(vb), _ptr(gb), touched.data_ptr(), lr,
                                         beta1, beta2, eps, weight_decay, step, st), 'hsk_adamw_rows_lazy')


def adamw_consts(lr, beta1, beta2, eps, weight_decay, step: int, out_host: torch.Tensor):
    """Fill the 8 fp32 step scalars into a (pinned) HOST tensor."""
    if out_host.is_cuda or out_host.dtype != torch.float32 or out_host.numel() < 8:
        raise HskError('adamw_consts: out_host must be a host fp32 tensor with >= 8 elements')
    _check(lib().hsk_adamw_consts(lr, beta1, beta2, eps, weight_decay, step, out_host.data_ptr()), 'hsk_adamw_consts')


def adamw_dense_graph(p, m, v, g, consts_dev, decoupled: bool = True, adam_l2: bool = False, zero_grad: bool = True):
    for n, t in (('p', p), ('m', m), ('v', v), ('g', g), ('consts_dev', consts_dev)):
        _req(t, torch.float32, n)
    with _on_device_of(p, m, v, g, consts_dev) as st:
        _check(lib().hsk_adamw_dense_graph(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), p.numel(),
                                           consts_dev.data_ptr(), int(decoupled), int(adam_l2), int(zero_grad), st),
               'hsk_adamw_dense_graph')


def sample_negatives(u_idx, pos_idx, n_neg: int, n_items: int, n_users: int, csr_indptr, csr_indices, seed: int,
                     step: int, i_idx, distinct_in_row: bool = True, status=None, pop_cdf=None):
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx')
    _req(csr_indptr, torch.int64, 'csr_indptr'); _req(csr_indices, torch.int32, 'csr_indices')
    if pos_idx is not None:
        _req(pos_idx, torch.int64, 'pos_idx')
    B = u_idx.numel()
    if tuple(i_idx.shape) != (B, n_neg + 1):
        raise HskError(f'i_idx must be [{B}, {n_neg + 1}]')
    with _on_device_of(u_idx, pos_idx, csr_indptr, csr_indices, i_idx, status, pop_cdf) as st:
        _check(lib().hsk_sample_negatives(u_idx.data_ptr(), _ptr(pos_idx), B, n_neg, n_items, n_users, csr_indptr.data_ptr(),
                                          csr_indices.data_ptr(), seed & 0xFFFFFFFFFFFFFFFF, step, int(distinct_in_row),
                                          _ptr(pop_cdf), i_idx.data_ptr(), _ptr(status), st), 'hsk_sample_negatives')


# ---- evaluator ----
def eval_topk_scratch_bytes(Be: int, n_local_items: int, k: int) -> int:
    return int(lib().hsk_eval_topk_scratch_bytes(Be, n_local_items, k))


def eval_topk(tables: MfTables, u_idx, k: int, top_scores, top_ids, scratch, excl_indptr=None, excl_indices=None,
              id_offset: int = 0, id_stride: int = 1, status=None, u_rows=None, n_users_global: int = 0):
    _req(u_idx, torch.int64, 'u_idx'); _req(top_scores, torch.float32, 'top_scores'); _req(top_ids, torch.int32, 'top_ids')
    if excl_indptr is not None:
        _req(excl_indptr, torch.int64, 'excl_indptr'); _req(excl_indices, torch.int32, 'excl_indices')
    Be = u_idx.numel()
    if u_rows is not None:
        _req(u_rows, torch.int64, 'u_rows')
    with _on_device_of(u_idx, top_scores, top_ids, scratch, excl_indptr, excl_indices, status, u_rows) as st:
        _check(lib().hsk_eval_topk(C.byref(tables), u_idx.data_ptr(), _ptr(u_rows), n_users_global, Be, id_offset, id_stride,
                                   _ptr(excl_indptr), _ptr(excl_indices), k, top_scores.data_ptr(), top_ids.data_ptr(),
                                   scratch.data_ptr(), scratch.numel() * scratch.element_size(), _ptr(status), st),
               'hsk_eval_topk')


def eval_tc_kpad(d: int, precision: int) -> int:
    return int(lib().hsk_eval_tc_kpad(d, precision))


def pack_rows(src, d: int, precision: int, row_idx=None, out=None, status=None):
    """fp32 table rows [n, ld] (optionally gathered by row_idx) -> packed [rows, kpad] bf16 / tf32 operand."""
    if not src.is_cuda or src.dtype != torch.float32 or src.dim() != 2 or src.stride(1) != 1:
        raise HskError('pack_rows: src must be a 2-D fp32 CUDA tensor with unit inner stride')
    kpad = eval_tc_kpad(d, precision)
    n_out = src.shape[0] if row_idx is None else row_idx.numel()
    dt = torch.float32 if precision == PRECISIONS['tf32'] else torch.bfloat16
    if out is None:
        out = torch.empty((n_out, kpad), dtype=dt, device=src.device)
    if row_idx is not None:
        _req(row_idx, torch.int64, 'row_idx')
    with _on_device_of(src, row_idx, out, status) as st:
        _check(lib().hsk_pack_rows(src.data_ptr(), src.stride(0), d, _ptr(row_idx), n_out, src.shape[0], out.data_ptr(),
                                   kpad, precision, _ptr(status), st), 'hsk_pack_rows')
    return out


def eval_topk_tc_scratch_bytes(Be: int, n_local_items: int, k: int) -> int:
    return int(lib().hsk_eval_topk_tc_scratch_bytes(Be, n_local_items, k))


def eval_topk_tc(Uq, Vq, precision: int, u_idx, n_users: int, k: int, top_scores, top_ids, scratch, Ub=None, Ib=None,
                 Gb=None, excl_indptr=None, excl_indices=None, id_offset: int = 0, id_stride: int = 1, status=None,
                 u_rows=None, variant: Optional[str] = None):
    _req(u_idx, torch.int64, 'u_idx'); _req(top_scores, torch.float32, 'top_scores'); _req(top_ids, torch.int32, 'top_ids')
    Be, kpad = Uq.shape
    with _on_device_of(Uq, Vq, u_idx, top_scores, top_ids, scratch, Ub, Ib, Gb, excl_indptr, excl_indices, status, u_rows) as st:
        _check(lib().hsk_eval_topk_tc_v(Uq.data_ptr(), Vq.data_ptr(), kpad, precision, _ptr(Ub), _ptr(Ib), _ptr(Gb),
                                        u_idx.data_ptr(), _ptr(u_rows), Be, n_users, Vq.shape[0], id_offset, id_stride,
                                        _ptr(excl_indptr), _ptr(excl_indices), k, top_scores.data_ptr(), top_ids.data_ptr(),
                                        scratch.data_ptr(), scratch.numel() * scratch.element_size(), _ptr(status),
                                        EVAL_TC_VARIANTS[variant or EVAL_TC_VARIANT], st), 'hsk_eval_topk_tc')


class ItemShards:
    """The item tables of every rank of a node as seen from THIS process (device addresses): packed tensor-core operands
    `Vq` [rows_q, kpad], fp32 rows `V` [rows_q, ld], item bias `Ib` [rows_q] (None: no bias), rank order.  Item id =
    q + n_shards * row."""

    def __init__(self, rows, Vq=None, V=None, Ib=None):
        self.n = len(rows)
        if not 1 <= self.n <= MAX_PEERS:
            raise ValueError(f'1..{MAX_PEERS} item shards, got {self.n}')
        self.rows = (C.c_int64 * self.n)(*[int(r) for r in rows])
        arr = lambda ptrs: (C.c_void_p * self.n)(*[int(p) for p in ptrs]) if ptrs is not None else None
        self.Vq, self.V, self.Ib = arr(Vq), arr(V), arr(Ib)


def eval_topk_tc_shards_scratch_bytes(Be: int, shards: ItemShards, k: int) -> int:
    return int(lib().hsk_eval_topk_tc_shards_scratch_bytes(Be, shards.rows, shards.n, k))


def eval_topk_tc_shards(Uq, shards: ItemShards, precision: int, u_idx, n_users: int, k: int, top_scores, top_ids, scratch, Ub=None,
                        Gb=None, excl_indptr=None, excl_indices=None, status=None, u_rows=None):
    """hsk_eval_topk_tc_shards: tcgen05 scoring of the batch against ALL item shards (peer-mapped packed tables)."""
    _req(u_idx, torch.int64, 'u_idx'); _req(top_scores, torch.float32, 'top_scores'); _req(top_ids, torch.int32, 'top_ids')
    with _on_device_of(Uq, u_idx, top_scores, top_ids, scratch, Ub, Gb, excl_indptr, excl_indices, status, u_rows) as st:
        _check(lib().hsk_eval_topk_tc_shards(Uq.data_ptr(), shards.Vq, shards.rows, shards.Ib, shards.n, Uq.shape[1], precision,
                                             _ptr(Ub), _ptr(Gb), u_idx.data_ptr(), _ptr(u_rows), u_idx.numel(), n_users,
                                             _ptr(excl_indptr), _ptr(excl_indices), k, top_scores.data_ptr(), top_ids.data_ptr(),
                                             scratch.data_ptr(), scratch.numel() * scratch.element_size(), _ptr(status), st),
               'hsk_eval_topk_tc_shards')


def rescore_topk_shards(tables: MfTables, shards: ItemShards, u_rows, cand_ids, k: int, top_scores, top_ids, status=None,
                        cand_scores=None):
    """hsk_rescore_topk_shards: fp32 re-scoring with the item rows read from the (peer-mapped) shards."""
    _req(u_rows, torch.int64, 'u_rows'); _req(cand_ids, torch.int32, 'cand_ids')
    Be, n_cand = cand_ids.shape
    with _on_device_of(u_rows, cand_ids, top_scores, top_ids, status, cand_scores) as st:
        _check(lib().hsk_rescore_topk_shards(C.byref(tables), shards.V, shards.rows, shards.Ib, shards.n, u_rows.data_ptr(), Be,
                                             cand_ids.data_ptr(), _ptr(cand_scores), n_cand, k, top_scores.data_ptr(),
                                             top_ids.data_ptr(), _ptr(status), st), 'hsk_rescore_topk_shards')


def rescore_topk(tables: MfTables, u_rows, cand_ids, k: int, top_scores, top_ids, id_offset: int = 0, id_stride: int = 1,
                 status=None, cand_scores=None):
    """fp32 re-scoring of tensor-core candidates: cand_ids int32 [Be, n_cand <= 128] -> exact top-k of the candidates;
    cand_scores (the low-precision scores): -inf marks an excluded item, which stays -inf."""
    _req(u_rows, torch.int64, 'u_rows'); _req(cand_ids, torch.int32, 'cand_ids')
    _req(top_scores, torch.float32, 'top_scores'); _req(top_ids, torch.int32, 'top_ids')
    Be, n_cand = cand_ids.shape
    if tuple(top_scores.shape) != (Be, k) or tuple(top_ids.shape) != (Be, k):
        raise HskError(f'rescore_topk: outputs must be [{Be}, {k}]')
    if cand_scores is not None:
        _req(cand_scores, torch.float32, 'cand_scores')
        if cand_scores.shape != cand_ids.shape:
            raise HskError('rescore_topk: cand_scores must have the shape of cand_ids')
    with _on_device_of(u_rows, cand_ids, cand_scores, top_scores, top_ids, status) as st:
        _check(lib().hsk_rescore_topk(C.byref(tables), u_rows.data_ptr(), Be, id_offset, id_stride, cand_ids.data_ptr(),
                                      _ptr(cand_scores), n_cand, k, top_scores.data_ptr(), top_ids.data_ptr(), _ptr(status),
                                      st), 'hsk_rescore_topk')


def rescore_scores(tables: MfTables, u_rows, cand_ids, out_scores, id_offset: int = 0, id_stride: int = 1, status=None):
    """Positional fp32 scores of the candidates this shard owns (-inf for the others): item-sharded evaluation."""
    _req(u_rows, torch.int64, 'u_rows'); _req(cand_ids, torch.int32, 'cand_ids'); _req(out_scores, torch.float32, 'out_scores')
    Be, n_cand = cand_ids.shape
    if tuple(out_scores.shape) != (Be, n_cand):
        raise HskError(f'rescore_scores: out_scores must be [{Be}, {n_cand}]')
    with _on_device_of(u_rows, cand_ids, out_scores, status) as st:
        _check(lib().hsk_rescore_scores(C.byref(tables), u_rows.data_ptr(), Be, id_offset, id_stride, cand_ids.data_ptr(), n_cand,
                                        out_scores.data_ptr(), _ptr(status), st), 'hsk_rescore_scores')


def topk_combine(scores, ids, k: int, out_scores, out_ids, cand_scores=None):
    """scores [G, rows, n_cand] (finite where shard g owns the item), ids [rows, n_cand] -> the k best per row;
    cand_scores [rows, n_cand] (the merged low-precision scores): -inf marks an excluded item, which stays -inf."""
    _req(scores, torch.float32, 'scores'); _req(ids, torch.int32, 'ids')
    _req(out_scores, torch.float32, 'out_scores'); _req(out_ids, torch.int32, 'out_ids')
    G, rows, n_cand = scores.shape
    if tuple(ids.shape) != (rows, n_cand) or tuple(out_scores.shape) != (rows, k) or tuple(out_ids.shape) != (rows, k):
        raise HskError('topk_combine: ids must be [rows, n_cand], outputs [rows, k]')
    if cand_scores is not None:
        _req(cand_scores, torch.float32, 'cand_scores')
        if cand_scores.shape != ids.shape:
            raise HskError('topk_combine: cand_scores must have the shape of ids')
    with _on_device_of(scores, ids, cand_scores, out_scores, out_ids) as st:
        _check(lib().hsk_topk_combine(scores.data_ptr(), ids.data_ptr(), _ptr(cand_scores), G, rows, n_cand, k,
                                      out_scores.data_ptr(), out_ids.data_ptr(), st), 'hsk_topk_combine')


def topk_merge(scores, ids, out_scores, out_ids):
    _req(scores, torch.float32, 'scores'); _req(ids, torch.int32, 'ids')
    _req(out_scores, torch.float32, 'out_scores'); _req(out_ids, torch.int32, 'out_ids')
    G, rows, k = scores.shape
    with _on_device_of(scores, ids, out_scores, out_ids) as st:
        _check(lib().hsk_topk_merge(scores.data_ptr(), ids.data_ptr(), G, rows, k, out_scores.data_ptr(),
                                    out_ids.data_ptr(), st), 'hsk_topk_merge')


def topk_dense(logits, k: int, out_scores, out_ids):
    _req(logits, torch.float32, 'logits', contiguous=False)
    if logits.dim() != 2 or logits.stride(1) != 1:
        raise HskError('logits must be 2-D with unit inner stride')
    _req(out_scores, torch.float32, 'out_scores'); _req(out_ids, torch.int32, 'out_ids')
    rows, cols = logits.shape
    with _on_device_of(logits, out_scores, out_ids) as st:
        _check(lib().hsk_topk_dense(logits.data_ptr(), rows, cols, logits.stride(0), k, out_scores.data_ptr(),
                                    out_ids.data_ptr(), st), 'hsk_topk_dense')


def topk_tag_means(top_ids, item_tag, ks, out=None, status=None):
    """hsk_topk_tag_means: [B, len(ks), T] mean tag rows of the first k ranked items, for every k in ks."""
    _req(top_ids, torch.int32, 'top_ids'); _req(item_tag, torch.float32, 'item_tag')
    B, k_list = top_ids.shape
    n_items, T = item_tag.shape
    if out is None:
        out = torch.empty((B, len(ks), T), dtype=torch.float32, device=top_ids.device)
    arr = (C.c_int * len(ks))(*[int(k) for k in ks])
    with _on_device_of(top_ids, item_tag, out, status) as st:
        _check(lib().hsk_topk_tag_means(top_ids.data_ptr(), B, k_list, item_tag.data_ptr(), n_items, T, arr, len(ks), out.data_ptr(),
                                        _ptr(status), st), 'hsk_topk_tag_means')
    return out


def _ks_array(ks):
    return (C.c_int * len(ks))(*[int(k) for k in ks])


def rank_metrics(top_ids, ks, u_idx, lab_indptr, lab_indices, discount, sums, counts, user_group=None, n_groups=0,
                 per_user=None):
    _req(top_ids, torch.int32, 'top_ids'); _req(u_idx, torch.int64, 'u_idx')
    _req(lab_indptr, torch.int64, 'lab_indptr'); _req(lab_indices, torch.int32, 'lab_indices')
    _req(discount, torch.float32, 'discount'); _req(sums, torch.float64, 'sums'); _req(counts, torch.int64, 'counts')
    if user_group is not None:
        _req(user_group, torch.int32, 'user_group')
    Be, k_max = top_ids.shape
    with _on_device_of(top_ids, u_idx, lab_indptr, lab_indices, discount, sums, counts, user_group, per_user) as st:
        _check(lib().hsk_rank_metrics(top_ids.data_ptr(), Be, k_max, _ks_array(ks), len(ks), u_idx.data_ptr(),
                                      lab_indptr.data_ptr(), lab_indices.data_ptr(), _ptr(user_group), n_groups,
                                      discount.data_ptr(), _ptr(per_user), sums.data_ptr(), counts.data_ptr(), st),
               'hsk_rank_metrics')


def rank_metrics_dense(top_ids, ks, u_idx, y_true, discount, sums, counts, user_group=None, n_groups=0, per_user=None):
    _req(top_ids, torch.int32, 'top_ids'); _req(u_idx, torch.int64, 'u_idx'); _req(y_true, torch.float32, 'y_true')
    _req(discount, torch.float32, 'discount'); _req(sums, torch.float64, 'sums'); _req(counts, torch.int64, 'counts')
    if user_group is not None:
        _req(user_group, torch.int32, 'user_group')
    Be, k_max = top_ids.shape
    with _on_device_of(top_ids, u_idx, y_true, discount, sums, counts, user_group, per_user) as st:
        _check(lib().hsk_rank_metrics_dense(top_ids.data_ptr(), Be, k_max, _ks_array(ks), len(ks), u_idx.data_ptr(),
                                            y_true.data_ptr(), y_true.shape[1], _ptr(user_group), n_groups,
                                            discount.data_ptr(), _ptr(per_user), sums.data_ptr(), counts.data_ptr(), st),
               'hsk_rank_metrics_dense')


# ---- deterministic mode (hsk_det.cu) ----
def det_scratch_bytes(B: int, N1: int, ld: int) -> int:
    return int(lib().hsk_det_scratch_bytes(B, N1, ld))


def _scratch_bytes(scratch) -> int:
    return scratch.numel() * scratch.element_size()


def mf_scatter_grads_det(tables: MfTables, grads: MfTables, u_idx, i_idx, dscores, scratch, status=None):
    """hsk_mf_scatter_grads_det: the touched rows of `grads` are STORED (fixed summation order, no atomics)."""
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(dscores, torch.float32, 'dscores')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, dscores, scratch, status) as st:
        _check(lib().hsk_mf_scatter_grads_det(C.byref(tables), C.byref(grads), u_idx.data_ptr(), i_idx.data_ptr(),
                                              dscores.data_ptr(), B, N1, scratch.data_ptr(), _scratch_bytes(scratch),
                                              _ptr(status), st), 'hsk_mf_scatter_grads_det')


def mf_train_fused_det(tables: MfTables, grads: MfTables, u_idx, i_idx, loss_kind: int, neg_shift: float, loss_accum,
                       scratch, scores_out=None, dscores_out=None, status=None, B_global: Optional[int] = None):
    """hsk_mf_train_fused_det: the fused step with per-sample dL/ds and a fixed-order scatter / loss sum.  `B_global`: the
    normalisers of a global batch this one is a share of (hsk_mf_train_fused_det_n, the sharded 'ordered' step)."""
    _req(u_idx, torch.int64, 'u_idx'); _req(i_idx, torch.int64, 'i_idx'); _req(loss_accum, torch.float64, 'loss_accum')
    B, N1 = i_idx.shape
    with _on_device_of(u_idx, i_idx, loss_accum, scratch, scores_out, dscores_out, status) as st:
        if B_global is None:
            _check(lib().hsk_mf_train_fused_det(C.byref(tables), C.byref(grads), u_idx.data_ptr(), i_idx.data_ptr(), B, N1,
                                                loss_kind, neg_shift, loss_accum.data_ptr(), _ptr(scores_out),
                                                _ptr(dscores_out), scratch.data_ptr(), _scratch_bytes(scratch), _ptr(status),
                                                st), 'hsk_mf_train_fused_det')
        else:
            _check(lib().hsk_mf_train_fused_det_n(C.byref(tables), C.byref(grads), u_idx.data_ptr(), i_idx.data_ptr(), B, N1,
                                                  B_global, loss_kind, neg_shift, loss_accum.data_ptr(), _ptr(scores_out),
                                                  _ptr(dscores_out), scratch.data_ptr(), _scratch_bytes(scratch), _ptr(status),
                                                  st), 'hsk_mf_train_fused_det_n')


def rec_loss_det(scores, labels, loss_kind: int, neg_shift: float, grad_scale: float, loss_accum, dscores, scratch,
                 shifted_out=None):
    """hsk_rec_loss_det: hsk_rec_loss with the per-row losses summed in a fixed order (scratch >= 8 * B bytes)."""
    _req(scores, torch.float32, 'scores'); _req(loss_accum, torch.float64, 'loss_accum'); _req(dscores, torch.float32, 'dscores')
    if labels is not None:
        _req(labels, torch.float64, 'labels')
    B, N1 = scores.shape
    with _on_device_of(scores, labels, loss_accum, dscores, shifted_out, scratch) as st:
        _check(lib().hsk_rec_loss_det(scores.data_ptr(), _ptr(labels), B, N1, loss_kind, neg_shift, grad_scale,
                                      loss_accum.data_ptr(), dscores.data_ptr(), _ptr(shifted_out), scratch.data_ptr(),
                                      _scratch_bytes(scratch), st), 'hsk_rec_loss_det')


def rank_metrics_sums_det(per_user, u_idx, sums, user_group=None, n_groups=0):
    """sums [(1 + n_groups), n_ks, 3] += fixed-order sums of per_user [Be, n_ks, 3] (hsk_rank_metrics_sums_det)."""
    _req(per_user, torch.float32, 'per_user'); _req(u_idx, torch.int64, 'u_idx'); _req(sums, torch.float64, 'sums')
    if user_group is not None:
        _req(user_group, torch.int32, 'user_group')
    Be, n_ks, _ = per_user.shape
    with _on_device_of(per_user, u_idx, sums, user_group) as st:
        _check(lib().hsk_rank_metrics_sums_det(per_user.data_ptr(), Be, n_ks, u_idx.data_ptr(), _ptr(user_group), n_groups,
                                               sums.data_ptr(), st), 'hsk_rank_metrics_sums_det')


# ---- packed validation: every active trial of a pack on one shared user batch ----
def eval_topk_pack_scratch_bytes(Be: int, n_items: int, k: int, n_active: int) -> int:
    return int(lib().hsk_eval_topk_pack_scratch_bytes(Be, n_items, k, n_active))


def eval_topk_pack(tables: MfTables, trial_stride: int, n_trials: int, active, u_idx, k: int, top_scores, top_ids, scratch,
                   excl_indptr=None, excl_indices=None, status=None):
    """hsk_eval_topk_pack: tables = trial 0's, trial j's at + j * trial_stride elements; top_scores / top_ids
    [n_active, Be, k]."""
    _req(u_idx, torch.int64, 'u_idx'); _req(active, torch.int32, 'active')
    _req(top_scores, torch.float32, 'top_scores'); _req(top_ids, torch.int32, 'top_ids')
    if excl_indptr is not None:
        _req(excl_indptr, torch.int64, 'excl_indptr'); _req(excl_indices, torch.int32, 'excl_indices')
    n_active, Be = active.numel(), u_idx.numel()
    for name, t in (('top_scores', top_scores), ('top_ids', top_ids)):
        if t.numel() != n_active * Be * k:
            raise HskError(f'{name} must be [n_active, Be, k] = [{n_active}, {Be}, {k}]')
    with _on_device_of(u_idx, active, top_scores, top_ids, scratch, excl_indptr, excl_indices, status) as st:
        _check(lib().hsk_eval_topk_pack(C.byref(tables), trial_stride, n_trials, active.data_ptr(), n_active, u_idx.data_ptr(), Be,
                                        _ptr(excl_indptr), _ptr(excl_indices), k, top_scores.data_ptr(), top_ids.data_ptr(),
                                        scratch.data_ptr(), _scratch_bytes(scratch), _ptr(status), st), 'hsk_eval_topk_pack')


def rank_metrics_pack(top_ids, ks, u_idx, lab_indptr, lab_indices, discount, active, sums, counts, user_group=None,
                      n_groups=0, per_user=None, status=None):
    """hsk_rank_metrics_pack: top_ids [n_active, Be, k_max]; sums fp64 [n_trials, 1 + n_groups, n_ks, 3], counts int64
    [n_trials, 1 + n_groups]; per_user (optional) [n_active, Be, n_ks, 3]."""
    _req(top_ids, torch.int32, 'top_ids'); _req(u_idx, torch.int64, 'u_idx'); _req(active, torch.int32, 'active')
    _req(lab_indptr, torch.int64, 'lab_indptr'); _req(lab_indices, torch.int32, 'lab_indices')
    _req(discount, torch.float32, 'discount'); _req(sums, torch.float64, 'sums'); _req(counts, torch.int64, 'counts')
    if user_group is not None:
        _req(user_group, torch.int32, 'user_group')
    if per_user is not None:
        _req(per_user, torch.float32, 'per_user')
    n_active, Be, k_max = top_ids.shape
    if n_active != active.numel():
        raise HskError(f'top_ids holds {n_active} trials, active lists {active.numel()}')
    n_trials = sums.shape[0]
    if sums.shape != (n_trials, 1 + n_groups, len(ks), 3) or counts.shape != (n_trials, 1 + n_groups):
        raise HskError(f'sums / counts must be [n_trials, 1 + n_groups, n_ks, 3] / [n_trials, 1 + n_groups] with n_groups = '
                       f'{n_groups}, n_ks = {len(ks)}')
    if per_user is not None and per_user.shape != (n_active, Be, len(ks), 3):
        raise HskError(f'per_user must be [n_active, Be, n_ks, 3] = [{n_active}, {Be}, {len(ks)}, 3]')
    with _on_device_of(top_ids, u_idx, active, lab_indptr, lab_indices, discount, sums, counts, user_group, per_user,
                       status) as st:
        _check(lib().hsk_rank_metrics_pack(top_ids.data_ptr(), Be, k_max, _ks_array(ks), len(ks), u_idx.data_ptr(),
                                           lab_indptr.data_ptr(), lab_indices.data_ptr(), _ptr(user_group), n_groups,
                                           discount.data_ptr(), n_trials, active.data_ptr(), n_active, _ptr(per_user),
                                           sums.data_ptr(), counts.data_ptr(), _ptr(status), st), 'hsk_rank_metrics_pack')


def rank_metrics_sums_det_pack(per_user, u_idx, batch: int, active, sums, user_group=None, n_groups=0, status=None):
    """hsk_rank_metrics_sums_det_pack: sums [n_trials, 1 + n_groups, n_ks, 3] += per trial, batch by batch in order, the
    fixed-order sums of per_user [n_active, Be, n_ks, 3]."""
    _req(per_user, torch.float32, 'per_user'); _req(u_idx, torch.int64, 'u_idx'); _req(active, torch.int32, 'active')
    _req(sums, torch.float64, 'sums')
    if user_group is not None:
        _req(user_group, torch.int32, 'user_group')
    n_active, Be, n_ks, _ = per_user.shape
    if n_active != active.numel():
        raise HskError(f'per_user holds {n_active} trials, active lists {active.numel()}')
    n_trials = sums.shape[0]
    if sums.shape != (n_trials, 1 + n_groups, n_ks, 3):
        raise HskError(f'sums must be [n_trials, 1 + n_groups, n_ks, 3] with n_groups = {n_groups}, n_ks = {n_ks}')
    with _on_device_of(per_user, u_idx, active, sums, user_group, status) as st:
        _check(lib().hsk_rank_metrics_sums_det_pack(per_user.data_ptr(), Be, batch, n_ks, u_idx.data_ptr(), _ptr(user_group),
                                                    n_groups, n_trials, active.data_ptr(), n_active, sums.data_ptr(),
                                                    _ptr(status), st), 'hsk_rank_metrics_sums_det_pack')
