"""CPU: the order contract of the sharded 'ordered' step (include/hassaku_b200.h) as restated by
tests/sharded_det_oracle.py (sharded_scatter_grads), and the host logic of ShardedMF._ordered_body at world 2 and 3 in the in-process
world of test_gpu_sharded_world.py, with the arithmetic plugged in from the numpy oracle."""
import numpy as np
import pytest
import torch

from hsk_testutil import ROOT  # noqa: F401
from oracle import det_oracle as D
from sharded_det_oracle import sharded_scatter_grads
from test_gpu_sharded_world import LOSS_CASES, _check_training, _Snapshots, world_of  # noqa: F401
from test_sharded_gloo import TorchRefOps


class OracleOps(TorchRefOps):
    """TorchRefOps plus the two operations of the ordered exchange, restated from the order contract: dL/ds from torch
    autograd, the per-rank scatter from det_oracle.scatter_grads (rows STORED), the rank-ordered composition at the owner."""

    def det_scratch_bytes(self, B, N1, ld):
        return 16

    def train_fused_det(self, lay, arena, g_arena, Vc, Ibc, gVc, gIbc, u_local, compact_idx, B_global, kind, shift,
                        loss_accum, scratch, dscores_out=None):
        B, N1 = compact_idx.shape
        if B == 0:
            return
        Uw, _, Ub, _, Gb = lay.views(arena)
        gU, _, gUb, _, gGb = lay.views(g_arena)
        s = (Uw[u_local][:, None, :] * Vc[:, :lay.d][compact_idx]).sum(-1)
        if Ub is not None:
            s = s + Ub.view(-1)[u_local][:, None]
        if Ibc is not None:
            s = s + Ibc[compact_idx]
        if Gb is not None:
            s = s + Gb
        s = s.detach().requires_grad_()
        if kind == 0:
            loss = (-torch.nn.functional.logsigmoid(s[:, :1] - s[:, 1:])).double().sum() / (B_global * (N1 - 1))
        elif kind == 1:
            s2 = torch.cat([s[:, :1], s[:, 1:] + shift], 1)
            loss = (-s2[:, 0] + torch.logsumexp(s2, -1)).double().sum() / B_global
        else:
            y = torch.zeros_like(s)
            y[:, 0] = 1.
            loss = torch.nn.functional.binary_cross_entropy_with_logits(s, y, reduction='sum').double() / (B_global * N1)
        loss.backward()
        ds = s.grad.float()
        if dscores_out is not None:
            dscores_out.copy_(ds)
        g = D.scatter_grads(Uw.numpy(), Vc[:, :lay.d].numpy(), u_local.numpy(), compact_idx.numpy(), ds.numpy(),
                            (Ub is not None, Ibc is not None, Gb is not None))
        touched_u = np.unique(u_local.numpy())
        gU[touched_u] = torch.from_numpy(g['gU'][touched_u])
        touched_i = np.unique(compact_idx.numpy())
        gVc[touched_i, :lay.d] = torch.from_numpy(g['gV'][touched_i])
        if Ub is not None:
            gUb.view(-1)[touched_u] = torch.from_numpy(g['gUb'][touched_u])
        if Ibc is not None:
            gIbc[touched_i] = torch.from_numpy(g['gIb'][touched_i])
        if Gb is not None:
            gGb.copy_(torch.from_numpy(g['gGb']))
        loss_accum += loss.detach()

    def unpack_ordered(self, inp, rows, world, capq, gV2d, gIb, stamps, step, step_dev):
        ld = gV2d.shape[1]
        written = set()
        for q in range(world):
            for k in range(capq):
                r = int(rows[q, k])
                if r < 0:
                    continue
                b = inp[q].view(-1)[capq * ld + k]
                if r in written:
                    gV2d[r] = gV2d[r] + inp[q, k]
                    if gIb is not None:
                        gIb[r] = gIb[r] + b
                else:
                    gV2d[r] = inp[q, k]
                    if gIb is not None:
                        gIb[r] = b
                    written.add(r)
                stamps[r] = 1 + step % 255


class _OracleSnap(_Snapshots, OracleOps):
    pass


@pytest.mark.parametrize('ub,ib,gb', [(False, False, False), (True, True, True)])
def test_sharded_oracle_at_world_1_is_the_single_gpu_contract(ub, ib, gb):
    rng = np.random.RandomState(3)
    U, I, d, B, N1 = 37, 300, 12, 90, 13
    Uw = rng.standard_normal((U, d)).astype(np.float32)
    Vw = rng.standard_normal((I, d)).astype(np.float32)
    u = rng.randint(0, U, B)
    i = rng.randint(0, I, (B, N1))
    i[:, 1] = 5                                   # a hot item: its bucket spans several chunks
    ds = rng.standard_normal((B, N1)).astype(np.float32)
    want = D.scatter_grads(Uw, Vw, u, i, ds, (ub, ib, gb))
    got = sharded_scatter_grads(Uw, Vw, u, i, [ds], 1, (ub, ib, gb))
    assert sorted(got) == sorted(want)
    for k, w in want.items():
        if w is None:
            assert got[k] is None, k
        else:
            assert got[k].dtype == np.float32 and np.array_equal(got[k].view(np.uint32), w.view(np.uint32)), k


def test_sharded_oracle_composes_the_ranks_in_rank_order():
    """Two ranks fetch item 0: its row is rank 0's contribution plus rank 1's; every other item and user row is one rank's
    value; the global bias is rank 0's sum plus rank 1's."""
    rng = np.random.RandomState(4)
    U, I, d, N1 = 6, 5, 4, 2
    Uw = rng.standard_normal((U, d)).astype(np.float32)
    Vw = rng.standard_normal((I, d)).astype(np.float32)
    u = np.array([0, 1, 2, 3])
    i = np.array([[0, 1], [0, 2], [3, 4], [0, 4]])
    ds = rng.standard_normal((4, N1)).astype(np.float32)
    got = sharded_scatter_grads(Uw, Vw, u, i, [ds[[0, 2]], ds[[1, 3]]], 2, (True, True, True))
    r0 = D.scatter_grads(Uw, Vw, u[[0, 2]], i[[0, 2]], ds[[0, 2]], (True, True, True))
    r1 = D.scatter_grads(Uw, Vw, u[[1, 3]], i[[1, 3]], ds[[1, 3]], (True, True, True))
    assert np.array_equal(got['gV'][0], r0['gV'][0] + r1['gV'][0])
    assert np.array_equal(got['gV'][4], r0['gV'][4] + r1['gV'][4])
    assert np.array_equal(got['gV'][2], r1['gV'][2]) and np.array_equal(got['gV'][3], r0['gV'][3])
    assert np.array_equal(got['gU'][[0, 2]], r0['gU'][[0, 2]]) and np.array_equal(got['gU'][[1, 3]], r1['gU'][[1, 3]])
    assert got['gGb'][0] == np.float32(r0['gGb'][0] + r1['gGb'][0])


@pytest.mark.parametrize('G,kind,flags', [(2, 'bpr', (False, True, False)), (3, 'bce', (True, True, True)),
                                          (3, 'sampled_softmax', (False, False, False))])
def test_ordered_body_in_process_world_on_cpu_matches_the_oracle(G, kind, flags, world_of):  # noqa: F811
    _check_training(world_of(G, 'cpu'), 'ordered', G, kind, flags, 6, _OracleSnap)


def test_ordered_step_entry_point_takes_an_empty_share_without_index_pointers():
    """A rank without samples in a step passes empty (null-pointer) index tensors to hsk_mf_train_fused_det_n: accepted
    at B = 0 (nothing is launched); B > 0 still needs them."""
    import ctypes
    from hassaku_b200 import _C
    lib = _C.lib()
    t = _C.MfTables(0x1000, 0x2000, None, None, None, 4, 4, 4, 4)
    g = _C.MfTables(0x3000, 0x4000, None, None, None, 4, 4, 4, 4)
    for B, rc in ((0, 0), (3, -1)):
        n = _C.det_scratch_bytes(B, 6, 4)
        assert lib.hsk_mf_train_fused_det_n(ctypes.byref(t), ctypes.byref(g), None, None, B, 6, 8, 0, 0.0, None, None, None,
                                            0x10000, n, None, None) == rc
    assert b'null' in lib.hsk_last_error()
