"""The sharded step and the sharded evaluation (hassaku_b200/sharded.py) at world sizes 2 to 8 on ONE GPU, every rank in
one process.

One Python thread per rank runs an unmodified ShardedMF(world=G, rank=r), each on its own CUDA stream (torch's current
stream is per thread and the library launches on it, so the ranks' kernels overlap).  The collectives go to `FakeDist`, an
in-process stand-in for torch.distributed, and the CUDA IPC calls of the peer exchange to stand-ins that hand out the
owner's own device address (an allocation cannot be IPC-mapped into the process that owns it), so `_peer_setup` and
`_map_peers` run unchanged.  What runs for real at G > 1: the routing, pack and unpack-add kernels (ragged shards, a rank
with an empty batch), the fused step with global normalisers (B_global > local B), the peer step kernel with owner = i % G
addressing (the division branch at G = 3, 5, 6, 7), system-scope reductions and stamp stores into other ranks' arenas with
several ranks adding into one owner row, the row-stamped AdamW, and the item-sharded (late re-score at tensor-core
precision, second-stream overlap), replicated and streamed evaluators.

Not covered here: the `*_graph` exchanges, which capture NCCL calls that an in-process stand-in cannot serve, and the
`hsk_peer_barrier` kernel (ranks spinning on one device could wait for a rank whose work is not enqueued yet), for which
`peer_barrier = 'nccl'` puts a stand-in all-reduce.  Both stay covered at world 1 (test_gpu_round2.py) and by the multi-GPU
tests (test_gpu_sharded.py).  The CPU test drives the same harness with the torch reference ops of test_sharded_gloo.py."""
import math
import threading

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import hassaku_b200.sharded
from hassaku_b200 import _C
from hassaku_b200.sharded import CudaOps, ShardedMF, partition_batch_by_user_owner
from hsk_testutil import ROOT  # noqa: F401
from test_sharded_gloo import TorchRefOps


# ---- in-process world ----------------------------------------------------------------------------------------------
class FakeDist:
    """What hassaku_b200.sharded calls of torch.distributed, served between the G rank threads of `run`.  A collective:
    synchronise the caller's stream, deposit a copy of the input, wait for every rank, compute this rank's output from all
    deposits (in rank order, so every rank reduces alike), synchronise, wait again (no deposit is replaced while a peer
    still reads it)."""
    ReduceOp = torch.distributed.ReduceOp

    def __init__(self, world: int, device, timeout: float = 120.0):
        self.world, self.device = world, torch.device(device)
        self._bar = threading.Barrier(world, timeout=timeout)
        self._slots = [None] * world
        self._tls = threading.local()

    def _sync(self):
        if self.device.type == 'cuda':
            torch.cuda.current_stream(self.device).synchronize()

    def _collective(self, value, out_fn):
        r = self._tls.rank
        self._slots[r] = value.clone() if isinstance(value, torch.Tensor) else value
        self._sync()
        self._bar.wait()
        out_fn(r, self._slots)
        self._sync()
        self._bar.wait()

    def all_to_all_single(self, out, inp, group=None):
        G = self.world

        def f(r, slots):
            for q in range(G):
                out.view(G, -1)[q].copy_(slots[q].reshape(G, -1)[r])
        self._collective(inp, f)

    def all_gather_into_tensor(self, out, inp, group=None):
        def f(r, slots):
            for q, x in enumerate(slots):
                out.view(self.world, -1)[q].copy_(x.reshape(-1))
        self._collective(inp, f)

    def reduce_scatter_tensor(self, out, inp, group=None):
        def f(r, slots):
            acc = slots[0].reshape(self.world, -1)[r].clone()
            for x in slots[1:]:
                acc += x.reshape(self.world, -1)[r]
            out.view(-1).copy_(acc)
        self._collective(inp, f)

    def all_reduce(self, t, op=ReduceOp.SUM, group=None):
        if op not in (self.ReduceOp.SUM, self.ReduceOp.MIN):
            raise NotImplementedError(f'all_reduce {op}')

        def f(r, slots):
            acc = slots[0].clone()
            for x in slots[1:]:
                acc = acc + x if op == self.ReduceOp.SUM else torch.minimum(acc, x)
            t.copy_(acc)
        self._collective(t, f)

    def all_gather_object(self, out_list, obj, group=None):
        self._collective(obj, lambda r, slots: out_list.__setitem__(slice(None), list(slots)))

    def barrier(self, group=None):
        self._collective(None, lambda r, slots: None)

    def get_backend(self, group=None):
        return 'nccl'        # the reduce-scatter branch the GPUs take

    def run(self, fn):
        """fn(rank) in one thread per rank (on CUDA each under its own stream); returns the ranks' results or re-raises the
        first failure.  A failing rank breaks the barrier, so the others leave their collectives at once."""
        G = self.world
        results, errors = [None] * G, [None] * G

        def main(r):
            self._tls.rank = r
            try:
                if self.device.type == 'cuda':
                    with torch.cuda.stream(torch.cuda.Stream(self.device)):
                        results[r] = fn(r)
                        self._sync()
                else:
                    results[r] = fn(r)
            except BaseException as ex:     # handed to the main thread
                errors[r] = ex
                self._bar.abort()

        threads = [threading.Thread(target=main, args=(r,), name=f'rank{r}') for r in range(G)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        failed = [e for e in errors if e is not None]
        if failed:
            raise next((e for e in failed if not isinstance(e, threading.BrokenBarrierError)), failed[0])
        return results


def _export_own_address(t):
    return t.data_ptr().to_bytes(8, 'little') + bytes(_C.PEER_HANDLE_BYTES - 8), 0


def _open_own_address(handle, device):
    return int.from_bytes(handle[:8], 'little')


@pytest.fixture
def world_of(monkeypatch):
    def make(G, device):
        fake = FakeDist(G, device)
        monkeypatch.setattr(hassaku_b200.sharded, 'dist', fake)
        monkeypatch.setattr(_C, 'peer_export', _export_own_address)
        monkeypatch.setattr(_C, 'peer_open', _open_own_address)
        monkeypatch.setattr(_C, 'peer_close', lambda base: None)
        return fake
    return make


# ---- training step ---------------------------------------------------------------------------------------------------
U, I, B, N = 61, 53, 40, 5          # prime table sizes: ragged shards at every G
HOT = 7
LR, WD = 1e-3, 1e-4
STEPS = 4
LOSS_CASES = [('bpr', (False, True, False)), ('sampled_softmax', (False, True, False)), ('bce', (True, True, True)),
              ('bce', (False, False, False))]


class _Snapshots:
    """Ops mixin: before each optimizer step, keep what the step produced — the parameters its gradient was taken at, the
    gradient arena after every exchange, the row stamps and the offsets of the row segments AdamW skips by stamp."""

    def bind(self, smf):
        self.smf, self.status, self.snaps = smf, smf.status, []

    def adamw(self, arena, m, v, g, segments, lr, wd, t, *a, **kw):
        self.snaps.append({'t': t, 'arena': arena.clone(), 'g': g.clone(), 'su': self.smf.stamp_users.clone(),
                           'si': self.smf.stamp_items.clone(), 'segs': [s[0] for s in segments]})
        super().adamw(arena, m, v, g, segments, lr, wd, t, *a, **kw)


class _CudaSnap(_Snapshots, CudaOps):
    pass


class _RefSnap(_Snapshots, TorchRefOps):
    pass


def _batches(G):
    """STEPS global batches: the last user and item ids (step 0); every rank with samples that all share one hot item, and
    duplicate items within rows (step 1); no sample for rank G - 1 (step 2)."""
    rng = np.random.RandomState(100 + G)
    out = []
    for s in range(STEPS):
        u = rng.randint(0, U, B)
        i = rng.randint(0, I, (B, N + 1))
        if s == 0:
            u[0], i[0, 1], i[1, 0] = U - 1, I - 1, I - 1
        elif s == 1:
            u[:G] = np.arange(G)
            i[:, 1] = HOT
            i[:, 3] = i[:, 2]
        elif s == 2:
            u[u % G == G - 1] -= 1
        out.append((torch.from_numpy(u.astype(np.int64)), torch.from_numpy(i.astype(np.int64))))
    return out


def _rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max())


def _full_tables(arenas, lays, G):
    """Gather per-rank arenas (parameters or gradients) into float64 full tables U, V, Ub, Ib, Gb (row x of rank q = id
    q + x G)."""
    out = {}
    for name, k, n in (('U', 0, U), ('V', 1, I), ('Ub', 2, U), ('Ib', 3, I)):
        views = [lay.views(a)[k] for lay, a in zip(lays, arenas)]
        if views[0] is None:
            continue
        full = torch.empty((n, views[0].shape[1]), dtype=torch.float64)
        for q in range(G):
            full[q::G] = views[q].double()
        out[name] = full
    gb = [lay.views(a)[4] for lay, a in zip(lays, arenas)]
    if gb[0] is not None:
        assert all(torch.equal(x, gb[0]) for x in gb), 'the replicated global bias differs between ranks'
        out['Gb'] = gb[0].double()
    return out


def _grads64(P, u, i, kind, shift):
    """float64 autograd of the union-batch loss with the normalisers of TorchRefOps.train_fused."""
    x = {k: v.clone().requires_grad_() for k, v in P.items()}
    s = (x['U'][u][:, None, :] * x['V'][i]).sum(-1)
    if 'Ub' in x:
        s = s + x['Ub'][u]
    if 'Ib' in x:
        s = s + x['Ib'][i][..., 0]
    if 'Gb' in x:
        s = s + x['Gb']
    nb, n1 = i.shape
    if kind == 'bpr':
        loss = -F.logsigmoid(s[:, :1] - s[:, 1:]).sum() / (nb * (n1 - 1))
    elif kind == 'sampled_softmax':
        s2 = torch.cat([s[:, :1], s[:, 1:] + shift], 1)
        loss = (torch.logsumexp(s2, -1) - s2[:, 0]).sum() / nb
    else:
        y = torch.zeros_like(s)
        y[:, 0] = 1.
        loss = F.binary_cross_entropy_with_logits(s, y, reduction='sum') / (nb * n1)
    loss.backward()
    return {k: v.grad for k, v in x.items()}


def _check_stamps(snaps, prev, lays, G, u, i, t):
    """Rows any rank touched carry stamp(t) at their owner, the others keep their stamp; AdamW reads the gradient of stamped
    rows only (hsk_adamw_dense_rows), so every row without stamp(t) must have an exactly zero gradient."""
    stamp = 1 + t % 255          # hsk_row_stamp
    for q, (sn, lay) in enumerate(zip(snaps, lays)):
        for off, key, n, ids in ((lay.off_U, 'su', lay.n_users, u), (lay.off_V, 'si', lay.n_items, i.reshape(-1))):
            if off not in sn['segs']:
                continue            # a table the optimizer streams densely carries no stamps
            st, before = sn[key][:n], prev[q][key][:n]
            touched = torch.zeros(n, dtype=torch.bool)
            touched[ids[ids % G == q] // G] = True
            assert bool((st[touched] == stamp).all()), (t, q, key, 'touched row without the step stamp')
            assert torch.equal(st[~touched], before[~touched]), (t, q, key, 'untouched row re-stamped')
            rows = sn['g'][off:off + n * lay.ld].view(n, lay.ld)
            assert float(rows[st != stamp].abs().sum()) == 0.0, (t, q, key, 'gradient in a row AdamW skips')


def _train_rank(r, fake, exchange, G, kind, flags, d, sd0, batches, shift, ops):
    dev = fake.device
    smf = ShardedMF(U, I, d, *flags, world=G, rank=r, device=dev, ops=ops)
    ops.bind(smf)
    smf.peer_barrier = 'nccl'
    smf.load_full_state_dict(sd0)
    losses = []
    for u, i in batches:
        ul, il = partition_batch_by_user_owner(u.to(dev), i.to(dev), G, r)
        smf.step(ul, il, B, kind, shift, LR, WD, exchange=exchange)
        losses.append(smf.pop_loss())
        smf.check_status()
    sd = smf.full_state_dict()
    g_max = float(smf.g.abs().max())
    smf.close()
    snaps = [{k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in sn.items()} for sn in ops.snaps]
    return {'losses': losses, 'sd': sd, 'g_max': g_max, 'snaps': snaps, 'layout': smf.layout}


def _check_training(fake, exchange, G, kind, flags, d, ops_cls):
    """Model: test_sharded_gloo.py::_worker.  G ranks free-run STEPS steps on their shares of the global batches; the
    oracle (torch.optim.AdamW on CPU) steps on the union batches."""
    from oracle import mf_oracle as O
    torch.manual_seed(7)
    ref = O.OracleMF(U, I, d, *flags)
    with torch.no_grad():
        for p in ref.parameters():
            p.copy_(torch.randn_like(p) * (0.7 * d ** -0.25 if p.dim() == 2 and p.shape[1] == d else 0.1))
    sd0 = {k: v.detach().clone() for k, v in ref.state_dict().items()}
    shift = math.log(I / N) if kind == 'sampled_softmax' else 0.0
    batches = _batches(G)
    tr = O.OracleTrainer(ref, kind, LR, WD, 'adamw', neg_train=N)
    ref_losses = [float(tr.step(u, i)['loss']) for u, i in batches]
    out = fake.run(lambda r: _train_rank(r, fake, exchange, G, kind, flags, d, sd0, batches, shift, ops_cls()))
    # per step: the loss summed over the ranks; after the run: the parameters, and nothing left in any gradient arena
    for r, o in enumerate(out):
        for s, (a, b) in enumerate(zip(o['losses'], ref_losses)):
            assert abs(a - b) <= 1e-5 * abs(b), (r, s, a, b)
        assert o['g_max'] == 0.0, r
    for n, p in ref.state_dict().items():
        err = _rel_err(out[0]['sd'][n], p)
        assert err < 1e-5 + 2e-3 * LR, (n, err)
    # every step's gradient, gathered from the owners, against float64; the stamps it was scattered with
    lays = [o['layout'] for o in out]
    prev = [{'su': torch.zeros_like(o['snaps'][0]['su']), 'si': torch.zeros_like(o['snaps'][0]['si'])} for o in out]
    for s, (u, i) in enumerate(batches):
        snaps = [o['snaps'][s] for o in out]
        assert [sn['t'] for sn in snaps] == [s + 1] * G
        want = _grads64(_full_tables([sn['arena'] for sn in snaps], lays, G), u, i, kind, shift)
        got = _full_tables([sn['g'] for sn in snaps], lays, G)
        assert sorted(got) == sorted(want)
        for name, w in want.items():
            err = _rel_err(got[name], w)
            assert err < 1e-5, (s, name, err)
        _check_stamps(snaps, prev, lays, G, u, i, s + 1)
        prev = snaps


def _train_cases():
    """Every (exchange, world) meets every loss case, and the embedding sizes rotate so that each (exchange, world) and each
    (exchange, loss case) meets every size: d 6 (ld 8, one float4 per lane of the quarter-warp kernel), 40, 128 (four
    float4 per lane, the peer limit), and for the staged exchanges 200 (the warp-per-row kernels)."""
    worlds = {'sparse': (2, 3, 5, 8), 'dense': (2, 3, 5, 8), 'peer': (2, 3, 5, 6, 7, 8)}
    dims = {'sparse': (6, 40, 128, 200), 'dense': (6, 40, 128, 200), 'peer': (6, 40, 128)}
    for ex in ('sparse', 'dense', 'peer'):
        for gi, G in enumerate(worlds[ex]):
            for li, (kind, flags) in enumerate(LOSS_CASES):
                d = dims[ex][(gi + li) % len(dims[ex])]
                fl = ''.join('T' if f else 'F' for f in flags)
                yield pytest.param(ex, G, kind, flags, d, id=f'{ex}-G{G}-{kind}-{fl}-d{d}')


@pytest.mark.gpu
@pytest.mark.parametrize('exchange,G,kind,flags,d', list(_train_cases()))
def test_sharded_step_at_world_G_matches_the_oracle(exchange, G, kind, flags, d, world_of):
    _check_training(world_of(G, 'cuda'), exchange, G, kind, flags, d, _CudaSnap)


@pytest.mark.parametrize('G,exchange,kind,flags', [(2, 'sparse', 'bpr', (False, True, False)),
                                                   (3, 'sparse', 'sampled_softmax', (False, True, False)),
                                                   (2, 'dense', 'bce', (True, True, True)),
                                                   (3, 'dense', 'bce', (False, False, False))])
def test_in_process_world_on_cpu_matches_the_oracle(G, exchange, kind, flags, world_of):
    """The harness itself: the torch reference ops on CPU, same checks as the GPU cases."""
    _check_training(world_of(G, 'cpu'), exchange, G, kind, flags, 6, _RefSnap)


@pytest.mark.parametrize('n_users,n_items', [(5, 53), (61, 6)])
def test_fewer_rows_than_ranks_is_rejected_at_construction(n_users, n_items):
    with pytest.raises(ValueError, match=r'at least one user row and one item row per rank.*>= world \(8\)'):
        ShardedMF(n_users, n_items, 6, world=8, rank=0, device='cpu', ops=TorchRefOps())


# ---- evaluation -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('prec', ['fp32', 'tf32', 'bf16'])
@pytest.mark.parametrize('G', [2, 3, 8])
def test_sharded_evaluation_at_world_G_equals_the_single_gpu_sweep(G, prec, world_of):
    """1201 users, 4007 items: ragged user and item shards at G = 2, 3, 8.  `evaluate` with bs users per rank and round:
    the last round holds one user of rank 0 and none of the other ranks."""
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.data.dataset import FullEvalDataset
    from hassaku_b200.data.synthetic import make_interactions
    from hassaku_b200.eval.eval import FullEvaluator, evaluate_recommender_algorithm
    nu, ni, d = 1201, 4007, 64
    bs = {2: 150, 3: 100, 8: 50}[G]
    assert (nu - 1) % (G * bs) == 0
    torch.manual_seed(5)
    single = SGDMatrixFactorization(nu, ni, d, True, True, True)
    with torch.no_grad():
        for p in single.parameters():
            p.copy_(torch.randn_like(p) * (0.4 if p.shape[-1] == d else 0.1))
    sd0 = {k: v.clone() for k, v in single.state_dict().items()}
    single.to('cuda')
    data = make_interactions(nu, ni, 40000, seed=2, n_user_groups=2)
    ds = FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, 2)

    class L:
        dataset, batch_size = ds, 256

    single.eval_precision = prec
    ref = evaluate_recommender_algorithm(single, L, FullEvaluator(True, 2, ds.user_to_user_group), 'cuda')
    fake = world_of(G, 'cuda')

    def rank(r):
        smf = ShardedMF(nu, ni, d, True, True, True, world=G, rank=r, device='cuda')
        smf.load_full_state_dict(sd0)
        ev = lambda: FullEvaluator(True, 2, ds.user_to_user_group)  # noqa: E731
        res = {'overlap': smf.evaluate(data.val, data.train, ev(), batch_size=bs, precision=prec),
               'serial': smf.evaluate(data.val, data.train, ev(), batch_size=bs, precision=prec, overlap=False),
               'replicated': smf.evaluate_replicated(data.val, data.train, ev(), batch_size=bs, precision=prec)}
        if prec != 'fp32':
            res['streamed'] = smf.evaluate_streamed(data.val, data.train, ev(), batch_size=bs, precision=prec)
        smf.check_status()
        smf.close()
        return res

    for r, res in enumerate(fake.run(rank)):
        for mode, got in res.items():
            assert sorted(got) == sorted(ref), (r, mode)
            for k_, v in ref.items():
                assert abs(got[k_] - v) <= 1e-9, (r, mode, k_, got[k_], v)
