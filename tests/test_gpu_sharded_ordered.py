"""GPU: the sharded step's ORDERED exchange (ShardedMF.step(exchange='ordered' / 'ordered_graph')), the deterministic
multi-GPU step, and sharded evaluation / ShardedTrainer.fit under torch.use_deterministic_algorithms(True).

World 2 to 8 run on one GPU, every rank a thread of one process (test_gpu_sharded_world.py's harness): the step against
the float64 oracle, the owners' gradients bit for bit against the order contract (tests/sharded_det_oracle.py:
sharded_scatter_grads), run-to-run identity with the ranks' timing varied.  World 1: bit identity with the single-GPU
deterministic step, the captured graph against the eager step.  Real NCCL: fit twice at world 1 (and 2 with two GPUs)."""
import math
import os
import random
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import hassaku_b200.sharded
from hassaku_b200.sharded import ShardedMF, partition_batch_by_user_owner
from hsk_testutil import ROOT  # noqa: F401
from sharded_det_oracle import sharded_scatter_grads
from test_gpu_sharded_world import (B, HOT, I, LOSS_CASES, LR, N, U, WD, FakeDist, _batches, _check_training, _CudaSnap,
                                    _full_tables, world_of)  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.fixture
def det_mode():
    """Call it to turn torch.use_deterministic_algorithms on; the previous state is restored afterwards."""
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    yield lambda: torch.use_deterministic_algorithms(True)
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def _bits(x):
    return np.ascontiguousarray(np.asarray(x, np.float32)).view(np.int32)


# ---- 1 + 2: world G on one GPU: float64 and the order contract ---------------------------------------------------------
def _capturing_ops(registry):
    class Capture(_CudaSnap):
        """_CudaSnap that also keeps every step's dL/ds of this rank's samples."""

        def bind(self, smf):
            super().bind(smf)
            self.ds = []
            registry[smf.spec.rank] = self

        def train_fused_det(self, lay, arena, g_arena, Vc, Ibc, gVc, gIbc, u_local, compact_idx, *a, dscores_out=None):
            ds = torch.full(compact_idx.shape, float('nan'), dtype=torch.float32, device=compact_idx.device)
            super().train_fused_det(lay, arena, g_arena, Vc, Ibc, gVc, gIbc, u_local, compact_idx, *a, dscores_out=ds)
            self.ds.append(ds.cpu())
    return Capture


def _ordered_cases():
    dims = (6, 40, 128, 200, 1024)
    for gi, G in enumerate((2, 3, 5, 8)):
        for li, (kind, flags) in enumerate(LOSS_CASES):
            d = dims[(gi + li) % len(dims)]
            fl = ''.join('T' if f else 'F' for f in flags)
            yield pytest.param(G, kind, flags, d, id=f'G{G}-{kind}-{fl}-d{d}')


@pytest.mark.parametrize('G,kind,flags,d', list(_ordered_cases()))
def test_ordered_step_at_world_G_matches_float64_and_the_order_contract(G, kind, flags, d, world_of):  # noqa: F811
    """Rank G - 1 gets an empty batch at step 2 and a hot item is shared by every rank at step 1 (_batches).  Then every
    step's gradient, gathered from the owners, bit-equals the contract fed the step's parameters and the captured dL/ds."""
    ranks = {}
    _check_training(world_of(G, 'cuda'), 'ordered', G, kind, flags, d, _capturing_ops(ranks))
    assert sorted(ranks) == list(range(G))
    lays = [ranks[r].smf.layout for r in range(G)]
    for s, (u, i) in enumerate(_batches(G)):
        snaps = [ranks[r].snaps[s] for r in range(G)]
        P = _full_tables([sn['arena'].cpu() for sn in snaps], lays, G)
        got = _full_tables([sn['g'].cpu() for sn in snaps], lays, G)
        assert all(ranks[r].ds[s].shape[0] == int((u % G == r).sum()) for r in range(G))
        want = sharded_scatter_grads(P['U'].float().numpy(), P['V'].float().numpy(), u.numpy(), i.numpy(),
                                     [ranks[r].ds[s].numpy() for r in range(G)], G, flags)
        for name, key in (('U', 'gU'), ('V', 'gV'), ('Ub', 'gUb'), ('Ib', 'gIb'), ('Gb', 'gGb')):
            if want[key] is None:
                assert name not in got, (s, name)
                continue
            np.testing.assert_array_equal(_bits(got[name].float().numpy().reshape(want[key].shape)), _bits(want[key]),
                                          err_msg=f'step {s} {name}')


# ---- 3: run-to-run identity under the switch, with the ranks' timing varied ----------------------------------------------
class DelayedDist(FakeDist):
    """FakeDist whose ranks arrive at every collective after a random per-rank delay (seeded)."""

    def __init__(self, world, device, seed):
        super().__init__(world, device)
        self._rngs = [random.Random(seed * 100 + r) for r in range(world)]

    def _collective(self, value, out_fn):
        time.sleep(self._rngs[self._tls.rank].random() * 0.004)
        super()._collective(value, out_fn)


def _initial_state(d, flags, seed=7):
    from oracle import mf_oracle as O
    torch.manual_seed(seed)
    ref = O.OracleMF(U, I, d, *flags)
    with torch.no_grad():
        for p in ref.parameters():
            p.copy_(torch.randn_like(p) * (0.7 * d ** -0.25 if p.dim() == 2 and p.shape[1] == d else 0.1))
    return {k: v.detach().clone() for k, v in ref.state_dict().items()}


def _run_world(fake, G, kind, flags, d, sd0, batches, exchange='ordered'):
    shift = math.log(I / N) if kind == 'sampled_softmax' else 0.0

    def rank(r):
        smf = ShardedMF(U, I, d, *flags, world=G, rank=r, device='cuda')
        smf.load_full_state_dict(sd0)
        losses = []
        for u, i in batches:
            ul, il = partition_batch_by_user_owner(u.cuda(), i.cuda(), G, r)
            smf.step(ul, il, B, kind, shift, LR, WD, exchange=exchange)
            losses.append(smf.pop_loss())
        smf.check_status()
        out = {k: getattr(smf, k).cpu() for k in ('arena', 'm', 'v', 'g', 'stamp_users', 'stamp_items')}
        out['losses'] = losses
        smf.close()
        return out
    return fake.run(rank)


@pytest.mark.parametrize('G,kind,flags,d', [(3, 'bce', (True, True, True), 40), (8, 'bpr', (False, True, False), 128),
                                            (5, 'sampled_softmax', (False, False, False), 200)])
def test_ordered_step_is_reproducible_across_runs_and_rank_timing(G, kind, flags, d, world_of, monkeypatch,  # noqa: F811
                                                                  det_mode):
    sd0 = _initial_state(d, flags)
    batches = _batches(G) * 2
    det_mode()
    first = _run_world(world_of(G, 'cuda'), G, kind, flags, d, sd0, batches)
    delayed = DelayedDist(G, 'cuda', seed=G)
    monkeypatch.setattr(hassaku_b200.sharded, 'dist', delayed)
    second = _run_world(delayed, G, kind, flags, d, sd0, batches)
    for r in range(G):
        for k in ('arena', 'm', 'v', 'g', 'stamp_users', 'stamp_items'):
            assert torch.equal(first[r][k].view(torch.int32) if first[r][k].is_floating_point() else first[r][k],
                               second[r][k].view(torch.int32) if second[r][k].is_floating_point() else second[r][k]), (r, k)
        assert first[r]['losses'] == second[r]['losses'], r
        assert first[r]['losses'] == first[0]['losses'], r          # every rank reports the same sum


# ---- 4: world 1 is the single-GPU deterministic step ---------------------------------------------------------------------
@pytest.mark.parametrize('kind,flags', LOSS_CASES)
def test_ordered_step_at_world_1_is_the_single_gpu_deterministic_step(kind, flags, det_mode):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import (RecBayesianPersonalizedRankingLoss, RecBinaryCrossEntropy,
                                               RecSampledSoftmaxLoss)
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    nu, ni, d, Bs, Ns, steps = 300, 2000, 40, 48, 9, 6
    torch.manual_seed(11)
    model = SGDMatrixFactorization(nu, ni, d, *flags)
    with torch.no_grad():
        for p in model.parameters():
            p.copy_(torch.randn_like(p) * (0.3 if p.shape[-1] == d else 0.1))
    sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model.to('cuda')
    loss = {'bpr': RecBayesianPersonalizedRankingLoss, 'bce': RecBinaryCrossEntropy,
            'sampled_softmax': lambda: RecSampledSoftmaxLoss(ni, 'uniform', Ns)}[kind]()
    opt = DenseAdam(model, lr=LR, weight_decay=WD)
    single = FusedMFTrainStep(model, loss, opt)
    smf = ShardedMF(nu, ni, d, *flags, world=1, rank=0, device='cuda')
    smf.load_full_state_dict(sd0)
    rng = np.random.RandomState(2)
    batches = [(torch.from_numpy(rng.randint(0, nu, Bs)).cuda(), torch.from_numpy(rng.randint(0, ni, (Bs, Ns + 1))).cuda())
               for _ in range(steps)]
    batches[1][1][:, 1] = 17                                    # a hot item over several chunks
    det_mode()
    for s, (u, i) in enumerate(batches):
        single(u, i)
        smf.step(u, i, Bs, kind, single.shift, LR, WD, exchange='ordered')
        a, b = single.pop_loss_sum(), smf.pop_loss()
        assert a == b, (s, a, b)
    smf.check_status()
    got = smf.full_state_dict()
    for k, v in model.state_dict().items():
        assert torch.equal(got[k].view(torch.int32), v.cpu().view(torch.int32)), k
    lay = smf.layout
    assert lay.n_total == model.layout.n_total
    for name, mine, theirs in (('m', smf.m, opt.m), ('v', smf.v, opt.v)):
        for j, (x, y) in enumerate(zip(lay.views(mine), model.layout.views(theirs))):
            if x is not None:
                assert torch.equal(x.view(torch.int32), y.view(torch.int32)), (name, j)


# ---- 5: the captured graph is the eager step ------------------------------------------------------------------------------
def test_ordered_graph_equals_eager_at_world_1_across_a_batch_shape_change(det_mode):
    nu, ni, d, Ns = 400, 3000, 64, 7
    flags = (True, True, True)
    torch.manual_seed(3)
    sd0 = {'user_embeddings.weight': torch.randn(nu, d) * 0.2, 'item_embeddings.weight': torch.randn(ni, d) * 0.2,
           'user_bias.weight': torch.randn(nu, 1) * 0.1, 'item_bias.weight': torch.randn(ni, 1) * 0.1,
           'global_bias': torch.randn(1) * 0.1}
    eager = ShardedMF(nu, ni, d, *flags, world=1, rank=0, device='cuda')
    graph = ShardedMF(nu, ni, d, *flags, world=1, rank=0, device='cuda')
    eager.load_full_state_dict(sd0)
    graph.load_full_state_dict(sd0)
    rng = np.random.RandomState(5)
    shapes = [64, 64, 40, 40, 64, 64, 40]        # the second 64-graph replays after the 40-graph ran
    det_mode()
    for s, b in enumerate(shapes):
        u = torch.from_numpy(rng.randint(0, nu, b)).cuda()
        i = torch.from_numpy(rng.randint(0, ni, (b, Ns + 1))).cuda()
        eager.step(u, i, b, 'bce', 0.0, LR, WD, exchange='ordered')
        graph.step(u, i, b, 'bce', 0.0, LR, WD, exchange='ordered_graph')
        assert eager.pop_loss() == graph.pop_loss(), s
        for k in ('arena', 'm', 'v', 'stamp_users', 'stamp_items'):
            x, y = getattr(eager, k), getattr(graph, k)
            assert torch.equal(x.view(torch.int32) if x.is_floating_point() else x,
                               y.view(torch.int32) if y.is_floating_point() else y), (s, k)
    eager.check_status()
    graph.check_status()
    graph.close()


# ---- 6: sharded evaluation under the switch ----------------------------------------------------------------------------
@pytest.mark.parametrize('prec', ['fp32', 'bf16'])
def test_sharded_evaluation_under_the_switch_is_reproducible(prec, world_of, det_mode):  # noqa: F811
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.data.dataset import FullEvalDataset
    from hassaku_b200.data.synthetic import make_interactions
    from hassaku_b200.eval.eval import FullEvaluator, evaluate_recommender_algorithm
    G, nu, ni, d, bs = 3, 1201, 4007, 64, 100
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
    det_mode()

    def rank(r):
        smf = ShardedMF(nu, ni, d, True, True, True, world=G, rank=r, device='cuda')
        smf.load_full_state_dict(sd0)
        ev = lambda: FullEvaluator(True, 2, ds.user_to_user_group)  # noqa: E731
        res = {}
        for rep in range(2):
            res[('sharded', rep)] = smf.evaluate(data.val, data.train, ev(), batch_size=bs, precision=prec)
            res[('replicated', rep)] = smf.evaluate_replicated(data.val, data.train, ev(), batch_size=bs, precision=prec)
            if prec != 'fp32':
                res[('streamed', rep)] = smf.evaluate_streamed(data.val, data.train, ev(), batch_size=bs, precision=prec)
        smf.check_status()
        smf.close()
        return res

    out = fake.run(rank)
    for r, res in enumerate(out):
        for (mode, rep), got in res.items():
            assert got == res[(mode, 0)] == out[0][(mode, 0)], (r, mode, rep)
            assert sorted(got) == sorted(ref), (r, mode)
            for k_, v in ref.items():
                assert abs(got[k_] - v) <= 1e-9, (r, mode, k_, got[k_], v)


# ---- 7: ShardedTrainer.fit under the switch, twice; the step on real NCCL -----------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker_fit_twice(rank, world, port, out_dir):
    import faulthandler
    faulthandler.dump_traceback_later(300, exit=True)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
        from hassaku_b200.data.dataloader import EvalLoader, NegativeSampler, TrainDataLoader
        from hassaku_b200.data.dataset import FullEvalDataset, TrainRecDataset
        from hassaku_b200.data.synthetic import make_interactions
        from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
        from hassaku_b200.train.sharded_trainer import ShardedTrainer
        nu, ni, d = 1500, 6000, 64
        dev = torch.device('cuda', rank)
        data = make_interactions(nu, ni, 60000, seed=4, n_user_groups=2)
        train_ds = TrainRecDataset.from_interactions(data.train, data.user_group, 2)
        val_ds = FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, 2)
        runs = []
        for rep in range(2):
            torch.use_deterministic_algorithms(False)
            torch.manual_seed(7)
            model = SGDMatrixFactorization(nu, ni, d, use_item_bias=True)
            loader = TrainDataLoader(NegativeSampler(train_ds, 10), train_ds, batch_size=512, shuffle=True, device=dev)
            conf = {'device': 'cuda', 'lr': 1e-2, 'wd': 1e-5, 'optimizer': 'adamw', 'n_epochs': 4,
                    'optimizing_metric': 'ndcg@10', 'max_patience': 3, 'model_path': os.path.join(out_dir, f'model{rep}'),
                    'seed': 3, 'sharded_exchange': 'ordered', 'running_settings': {'use_wandb': False, 'batch_verbose': False}}
            tr = ShardedTrainer(model, loader, EvalLoader(val_ds, 512), RecBayesianPersonalizedRankingLoss(), conf)
            assert tr._exchange_name() == 'ordered_graph'
            losses = []
            epoch = tr._train_one_epoch

            def record():
                out = epoch()
                losses.append(out['epoch_train_loss'])
                return out
            tr._train_one_epoch = record
            torch.use_deterministic_algorithms(True)
            best = tr.fit()
            torch.use_deterministic_algorithms(False)
            tr.close()
            runs.append((best, losses, {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}))
        (b0, l0, m0), (b1, l1, m1) = runs
        assert b0 == b1, (b0, b1)
        assert l0 == l1 and len(l0) >= 1, (l0, l1)
        assert all(torch.equal(m0[k].view(torch.int32), m1[k].view(torch.int32)) for k in m0)
        if rank == 0:
            c0 = torch.load(os.path.join(out_dir, 'model0', 'model.pth'))
            c1 = torch.load(os.path.join(out_dir, 'model1', 'model.pth'))
            assert sorted(c0) == sorted(c1)
            assert all(torch.equal(c0[k].view(torch.int32), c1[k].view(torch.int32)) for k in c0)
            open(os.path.join(out_dir, 'ok'), 'w').write('ok')
    finally:
        torch.use_deterministic_algorithms(False)
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [1, 2])
def test_sharded_trainer_fit_under_the_switch_is_reproducible(world, tmp_path):
    if torch.cuda.device_count() < world:
        pytest.skip(f'needs >= {world} GPUs')
    mp.spawn(_worker_fit_twice, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert (tmp_path / 'ok').exists()


def _worker_steps_twice(rank, world, port, out_dir):
    import faulthandler
    faulthandler.dump_traceback_later(300, exit=True)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        flags, d = (True, True, True), 40
        sd0 = _initial_state(d, flags)
        batches = _batches(world) * 3
        torch.use_deterministic_algorithms(True)
        runs = []
        for rep, exchange in enumerate(('ordered', 'ordered', 'ordered_graph', 'ordered_graph')):
            smf = ShardedMF(U, I, d, *flags, device='cuda')
            smf.load_full_state_dict(sd0)
            losses = []
            for s, (u, i) in enumerate(batches):
                if rep % 2 and rank == s % world:
                    time.sleep(0.01)                     # vary the ranks' arrival at the collectives
                ul, il = partition_batch_by_user_owner(u.cuda(), i.cuda(), world, rank)
                smf.step(ul, il, B, 'bce', 0.0, LR, WD, exchange=exchange)
                losses.append(smf.pop_loss())
            smf.check_status()
            runs.append((losses, smf.arena.cpu(), smf.m.cpu(), smf.v.cpu()))
            smf.close()
        for losses, p, m, v in runs[1:]:
            assert losses == runs[0][0]
            assert all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip((p, m, v), runs[0][1:]))
        if rank == 0:
            open(os.path.join(out_dir, 'ok'), 'w').write('ok')
    finally:
        torch.use_deterministic_algorithms(False)
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_ordered_step_is_reproducible_on_nccl(tmp_path):
    mp.spawn(_worker_steps_twice, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / 'ok').exists()
