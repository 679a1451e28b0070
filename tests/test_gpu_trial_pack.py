"""GPU: trial packs (hassaku_b200/train/trial_pack.py) — hsk_adamw_pack bitwise against torch.optim.AdamW / Adam per trial,
hsk_mf_train_fused_pack against the single-model step per trial, inactive trials untouched, status bits, guard words, and
PackedTrainer.fit against Trainer.fit (bitwise under torch.use_deterministic_algorithms(True))."""
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


# ---------------------------------------------------------------------------------------------------------------------
# packed optimizer
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('opt_name', ['adamw', 'adam'])
@pytest.mark.parametrize('form', ['dense', 'rows'])
def test_packed_adamw_bitwise_vs_torch_per_trial(opt_name, form):
    """3 active trials (distinct lr / wd, one wd = 0) + 1 inactive, 5 steps: each active trial's p / m / v equal
    torch.optim.AdamW / Adam on CUDA bit for bit; the inactive trial's p / m / v / g are not touched."""
    from hassaku_b200 import _C
    rows, ld, extra = 300, 12, 44            # one row segment [rows, ld] then a dense tail (bias-vector stand-in)
    stride = rows * ld + extra
    lrs, wds = [1e-3, 3e-4, 2e-2, 5e-3], [0.0, 4e-5, 1e-2, 1e-3]
    active_idx, M, steps = [0, 2, 3], 4, 5
    gen = torch.Generator().manual_seed(0)
    p0 = torch.randn(M, stride, generator=gen) * 0.05
    p0[:, :50] = -0.0                        # signed zeros: Adam(L2) with wd = 0 must keep -0 gradients -0
    grads = []
    for s in range(steps):
        g = torch.randn(M, stride, generator=gen) * 10 ** float(torch.randint(-6, 0, (1,), generator=gen))
        g[:, 50:100] = -0.0
        touched = torch.rand(rows, generator=gen) < 0.3
        if form == 'rows':                    # untouched rows of the segment have an all-zero gradient
            g[:, :rows * ld].view(M, rows, ld)[:, ~touched] = 0.0
        grads.append((g, touched))
    p, m, v, g = (torch.empty(M, stride, device='cuda') for _ in range(4))
    p.copy_(p0); m.zero_(); v.zero_()
    stamps = torch.zeros(rows, dtype=torch.uint8, device='cuda')
    active = torch.tensor(active_idx, dtype=torch.int32, device='cuda')
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    table = _C.adamw_consts_table(lrs, wds, 0.9, 0.999, 1e-8, 1, steps).cuda()
    g.copy_(grads[0][0])
    inactive_before = [_bits(x[1]) for x in (p, m, v, g)]
    for s, (gs, touched) in enumerate(grads, 1):
        for j in active_idx:
            g[j].copy_(gs[j])
        segs = ()
        if form == 'rows':
            _C.mark_rows(torch.nonzero(touched).flatten().cuda(), rows, stamps, step=s)
            segs = ((0, rows, ld, stamps),)
        _C.adamw_pack(p, m, v, g, active, table[s - 1], segs, step=s, adam_l2=opt_name == 'adam', status=status)
        for j in active_idx:
            assert float(g[j].abs().max()) == 0.0
    assert int(status.item()) == 0
    for x, b in zip((p, m, v), inactive_before[:3]):
        assert torch.equal(_bits(x[1]), b)
    assert torch.equal(_bits(g[1]), inactive_before[3])
    cls = torch.optim.AdamW if opt_name == 'adamw' else torch.optim.Adam
    for j in active_idx:
        q = torch.nn.Parameter(p0[j].clone().cuda())
        opt = cls([q], lr=lrs[j], weight_decay=wds[j])
        for gs, _ in grads:
            q.grad = gs[j].clone().cuda()
            opt.step()
        st = opt.state[q]
        for name, a, b in (('p', p[j], q), ('m', m[j], st['exp_avg']), ('v', v[j], st['exp_avg_sq'])):
            assert torch.equal(_bits(a), _bits(b)), f'trial {j} {name}: {(_bits(a) != _bits(b)).sum().item()} differ'


def test_packed_adamw_flags_a_bad_active_index():
    from hassaku_b200 import _C
    M, stride = 2, 64
    p, m, v, g = (torch.zeros(M, stride, device='cuda') for _ in range(4))
    g.fill_(1.0)
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    table = _C.adamw_consts_table([1e-3] * M, [0.0] * M, 0.9, 0.999, 1e-8, 1, 1).cuda()
    _C.adamw_pack(p, m, v, g, torch.tensor([0, 2], dtype=torch.int32, device='cuda'), table[0], status=status)
    assert int(status.item()) & _C.STATUS_BAD_INDEX
    assert float(g[0].abs().max()) == 0.0 and float(g[1].min()) == 1.0


# ---------------------------------------------------------------------------------------------------------------------
# packed step
# ---------------------------------------------------------------------------------------------------------------------
BIAS_COMBOS = [(False, False, False), (True, True, True), (False, True, False)]
D_LIST = [7, 64, 128, 402, 1024]


def _models(M, U, I, d, biases, seed0=10):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    out = []
    for j in range(M):
        mdl = SGDMatrixFactorization.on_device(U, I, d, *biases, device='cuda', seed=seed0 + j, std=(d ** -0.5, 0.1))
        if biases[2]:
            mdl.global_bias.data.fill_(0.05 * (j + 1))
        out.append(mdl)
    return out


def _loss(kind, N, I):
    from hassaku_b200.train.rec_losses import RecommenderSystemLossesEnum

    class _DS:
        n_items = I

    return RecommenderSystemLossesEnum[kind].value.build_from_conf({'train_neg_strategy': 'uniform', 'neg_train': N}, _DS())


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


@pytest.mark.parametrize('kind', ['bpr', 'sampled_softmax', 'bce'])
@pytest.mark.parametrize('d', D_LIST)
@pytest.mark.parametrize('B,M', [(1, 1), (64, 3), (8192, 17)])
def test_packed_step_matches_single_model_step(kind, d, B, M):
    """Every trial's loss and gradient tables against hsk_mf_train_fused of that trial alone, from the same state on the
    same batch (per-step gate), and its post-AdamW p / m / v, from that gradient, bitwise against hsk_adamw_dense(_rows);
    trial 1 (M > 1) is inactive and not written."""
    from hassaku_b200 import _C
    from hassaku_b200.train.optim import DenseAdam, stamp_segments
    from hassaku_b200.train.trial_pack import PackedMFTrainStep
    biases = BIAS_COMBOS[D_LIST.index(d) % 3]
    U, I, N = 700, 500, 4
    lrs = [1e-3 * (j + 1) for j in range(M)]
    wds = [0.0 if j % 2 == 0 else 1e-4 for j in range(M)]
    singles = _models(M, U, I, d, biases)
    packed = _models(M, U, I, d, biases)
    loss_fn = _loss(kind, N, I)
    step = PackedMFTrainStep(packed, loss_fn, lrs, wds, optimizer='adamw')
    inactive = [1] if M > 1 else []
    step.set_active([j not in inactive for j in range(M)])
    gen = torch.Generator(device='cuda')
    gen.manual_seed(3)
    u = torch.randint(0, U, (B,), device='cuda', generator=gen)
    i = torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)
    step.g.normal_(generator=gen)             # the inactive trial's gradient arena holds garbage that must stay as it is
    for j in range(M):
        if j not in inactive:
            step.g[j].zero_()
    before = [(_bits(step.p[j]), _bits(step.g[j])) for j in inactive]
    # fused step alone: gradients and losses
    _C.mf_train_fused_pack(step.tables, step.grad_tables, step.stride, M, step.active, u, i, step.kind, step.shift,
                           step.loss_accum, status=step.status)
    lay = packed[0].layout
    sums = step.loss_accum.tolist()
    for j in range(M):
        if j in inactive:
            continue
        opt = DenseAdam(singles[j], lr=lrs[j], weight_decay=wds[j])
        acc = torch.zeros(1, dtype=torch.float64, device='cuda')
        _C.mf_train_fused(singles[j]._tables(), opt.grad_tables, u, i, step.kind, step.shift, acc)
        assert abs(sums[j] - float(acc)) <= RTOL * abs(float(acc)), (j, sums[j], float(acc))
        # max-norm relative over the arena: the bias gradients of bpr are sums that cancel to rounding noise
        assert rel_err(step.g[j], opt.g) <= RTOL, (j, rel_err(step.g[j], opt.g))
        for name, a, b in zip(('gU', 'gV'), lay.views(step.g[j]), lay.views(opt.g)):
            assert rel_err(a, b) <= RTOL, (j, name, rel_err(a, b))
        # the optimizer on top, teacher-forced: both optimizers get the single model's gradient (two valid summation
        # orders of a nearly cancelling gradient move Adam's first update lr * g / (|g| + eps) by up to ~lr), so the
        # packed AdamW must reproduce the single-model rows / dense kernel bit for bit
        step.g[j].copy_(opt.g)
        segs, su, si = stamp_segments(lay, B, B * (N + 1), opt.stamp_users, opt.stamp_items)
        if segs:
            _C.mark_batch(u, i, U, I, su, si, step=1)
        opt._segments = segs
        opt.step_fused()
        singles[j]._opt = opt
    segs, su, si = stamp_segments(lay, B, B * (N + 1), step.stamp_users, step.stamp_items)
    if segs:
        _C.mark_batch(u, i, U, I, su, si, step=1)
    step.prepare(1)
    step.t = 1
    _C.adamw_pack(step.p, step.m, step.v, step.g, step.active, step._consts[0], segs, step=1, status=step.status)
    for j in range(M):
        if j in inactive:
            continue
        opt = singles[j]._opt
        for name, a, b in (('p', step.p[j], singles[j].arena), ('m', step.m[j], opt.m), ('v', step.v[j], opt.v)):
            assert torch.equal(_bits(a), _bits(b)), (j, name, int((_bits(a) != _bits(b)).sum()))
        assert float(step.g[j].abs().max()) == 0.0
    for j, (pb, gb) in zip(inactive, before):
        assert torch.equal(_bits(step.p[j]), pb) and torch.equal(_bits(step.g[j]), gb)
    step.check_status()


def test_packed_step_flags_bad_user_item_and_trial_indices():
    from hassaku_b200 import _C
    from hassaku_b200.train.trial_pack import PackedMFTrainStep
    U, I, d, B, N, M = 200, 150, 64, 32, 4, 3
    for kind in ('bpr', 'sampled_softmax', 'bce'):
        step = PackedMFTrainStep(_models(M, U, I, d, (True, True, True)), _loss(kind, N, I), [1e-3] * M, [0.0] * M)
        u = torch.randint(0, U, (B,), device='cuda')
        i = torch.randint(0, I, (B, N + 1), device='cuda')
        u_bad = u.clone(); u_bad[3] = U
        i_bad = i.clone(); i_bad[5, 2] = -1
        for uu, ii in ((u_bad, i), (u, i_bad)):
            step.step(uu, ii)
            with pytest.raises(IndexError):
                step.pop_loss_sums()
        step.step(u, i)
        step.pop_loss_sums()
        _C.mf_train_fused_pack(step.tables, step.grad_tables, step.stride, M,
                               torch.tensor([0, M], dtype=torch.int32, device='cuda'), u, i, step.kind, step.shift,
                               step.loss_accum, status=step.status)
        assert int(step.status.item()) & _C.STATUS_BAD_INDEX
        step.status.zero_()


class _Guarded:
    """A tensor carved out of a larger allocation whose margins hold a canary pattern (as test_gpu_round2.py's)."""
    PAD = 4096

    def __init__(self, shape, dtype, fill=None):
        n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
        n_al = (n + 255) // 256 * 256
        self.raw = torch.full((self.PAD + n_al + self.PAD,), 0xA5, dtype=torch.uint8, device='cuda')
        self.n = n
        self.t = self.raw[self.PAD:self.PAD + n].view(dtype).view(shape)
        if fill is not None:
            self.t.fill_(fill)

    def intact(self):
        return bool((self.raw[:self.PAD] == 0xA5).all()) and bool((self.raw[self.PAD + self.n:] == 0xA5).all())


def test_pack_kernels_do_not_write_outside_their_buffers():
    from hassaku_b200 import _C
    from hassaku_b200.algorithms.sgd_alg import ArenaLayout
    gen = torch.Generator(device='cuda'); gen.manual_seed(0)
    U, I, B, N, M = 901, 777, 300, 17, 3
    for d, kind in ((402, 0), (64, 1), (100, 2), (128, 0)):
        lay = ArenaLayout(U, I, d, True, True, True)
        guards = [_Guarded((M, lay.n_total), torch.float32, 0.0) for _ in range(4)]
        p, m, v, g = (x.t for x in guards)
        for j in range(M):
            for v_ in lay.views(p[j])[:4]:
                v_.copy_(torch.randn(v_.shape, device='cuda', generator=gen) * 0.1)
        acc = _Guarded((M,), torch.float64, 0.0)
        su, si = _Guarded((U,), torch.uint8, 0), _Guarded((I,), torch.uint8, 0)
        act = _Guarded((M,), torch.int32)
        act.t.copy_(torch.arange(M, dtype=torch.int32))
        cst = _Guarded((M, 8), torch.float32)
        cst.t.copy_(_C.adamw_consts_table([1e-3] * M, [1e-4] * M, 0.9, 0.999, 1e-8, 1, 1)[0])
        u = torch.randint(0, U, (B,), device='cuda', generator=gen)
        i = torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)
        _C.mf_train_fused_pack(lay.tables(p[0]), lay.tables(g[0]), lay.n_total, M, act.t, u, i, kind, 0.3, acc.t)
        _C.mark_batch(u, i, U, I, su.t, si.t, step=1)
        _C.adamw_pack(p, m, v, g, act.t, cst.t, [(lay.off_U, U, lay.ld, su.t), (lay.off_V, I, lay.ld, si.t)], step=1)
        _C.adamw_pack(p, m, v, g, act.t, cst.t)
        torch.cuda.synchronize()
        assert float(g.abs().max()) == 0.0
        for x in guards + [acc, su, si, act, cst]:
            assert x.intact(), d


# ---------------------------------------------------------------------------------------------------------------------
# end to end
# ---------------------------------------------------------------------------------------------------------------------
class _EvalLoader:
    def __init__(self, dataset, batch_size):
        self.dataset, self.batch_size = dataset, batch_size


def _data():
    from hassaku_b200.data.dataset import FullEvalDataset, TrainRecDataset
    from hassaku_b200.data.synthetic import make_interactions
    data = make_interactions(300, 200, 6000, seed=0, n_user_groups=2)
    tds = TrainRecDataset.from_interactions(data.train, data.user_group, 2)
    ds = FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, 2)
    return tds, ds


def _loader(tds):
    from hassaku_b200.data.dataloader import NegativeSampler, TrainDataLoader
    return TrainDataLoader(NegativeSampler(tds, n_neg=20), tds, batch_size=256, shuffle=True, seed=7)


def _model(seed):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    torch.manual_seed(seed)
    model = SGDMatrixFactorization(300, 200, 32, use_item_bias=True)
    with torch.no_grad():
        model.user_embeddings.weight.mul_(40.)
        model.item_embeddings.weight.mul_(40.)
    return model


# lr = 0 leaves the model where it is: its metric never improves, so with patience 1 it stops after one epoch
TRIALS = [dict(seed=1, lr=5e-3, wd=1e-5, n_epochs=3, max_patience=5),
          dict(seed=2, lr=2e-2, wd=0.0, n_epochs=2, max_patience=5),
          dict(seed=3, lr=0.0, wd=1e-4, n_epochs=4, max_patience=1)]


def _conf(tr, path, optimizer):
    return {'device': 'cuda', 'lr': tr['lr'], 'wd': tr['wd'], 'optimizer': optimizer, 'n_epochs': tr['n_epochs'],
            'optimizing_metric': 'ndcg@10', 'max_patience': tr['max_patience'], 'model_path': path,
            'running_settings': {'use_wandb': False, 'batch_verbose': False}}


@pytest.fixture
def det_mode():
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    yield lambda: torch.use_deterministic_algorithms(True)
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


@pytest.mark.parametrize('optimizer', ['adamw', 'adam'])
def test_packed_trainer_bitwise_equal_to_trainer_under_determinism(optimizer, det_mode):
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer import Trainer
    from hassaku_b200.train.trial_pack import PackedTrainer
    tds, ds = _data()
    det_mode()
    with tempfile.TemporaryDirectory() as tmp:
        paths = [os.path.join(tmp, f'pack{j}') for j in range(len(TRIALS))]
        for pth in paths:
            os.makedirs(pth)
        pt = PackedTrainer([_model(t['seed']) for t in TRIALS], _loader(tds), _EvalLoader(ds, 128),
                           RecBayesianPersonalizedRankingLoss(), [_conf(t, pth, optimizer) for t, pth in zip(TRIALS, paths)])
        got = pt.fit()
        got_sd = [torch.load(os.path.join(pth, 'model.pth'), map_location='cpu') for pth in paths]
        assert [len(x) for x in pt.epoch_losses] == [3, 2, 1]
        for j, t in enumerate(TRIALS):
            pth = os.path.join(tmp, f'single{j}')
            os.makedirs(pth)
            tr = Trainer(_model(t['seed']), _loader(tds), _EvalLoader(ds, 128), RecBayesianPersonalizedRankingLoss(),
                         _conf(t, pth, optimizer))
            logs = []
            tr._report = lambda log_dict, epoch: logs.append(dict(log_dict))
            want = tr.fit()
            want_sd = torch.load(os.path.join(pth, 'model.pth'), map_location='cpu')
            assert got[j] == want, j
            assert [x['epoch_train_loss'] for x in logs[1:]] == [x['epoch_train_loss'] for x in pt.epoch_losses[j]], j
            assert set(got_sd[j]) == set(want_sd)
            for k in want_sd:
                assert torch.equal(got_sd[j][k], want_sd[k]), (j, k)


def test_packed_trainer_default_mode_metrics_match_checkpoints():
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.eval.eval import FullEvaluator, evaluate_recommender_algorithm
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trial_pack import PackedTrainer
    tds, ds = _data()
    with tempfile.TemporaryDirectory() as tmp:
        paths = [os.path.join(tmp, f'pack{j}') for j in range(len(TRIALS))]
        for pth in paths:
            os.makedirs(pth)
        best = PackedTrainer([_model(t['seed']) for t in TRIALS], _loader(tds), _EvalLoader(ds, 128),
                             RecBayesianPersonalizedRankingLoss(), [_conf(t, pth, 'adamw') for t, pth in zip(TRIALS, paths)]).fit()
        for j, pth in enumerate(paths):
            model = SGDMatrixFactorization(300, 200, 32, use_item_bias=True)
            model.load_state_dict(torch.load(os.path.join(pth, 'model.pth'), map_location='cpu'))
            model.to('cuda')
            ev = FullEvaluator(aggr_by_group=True, n_groups=ds.n_user_groups, user_to_user_group=ds.user_to_user_group)
            fresh = evaluate_recommender_algorithm(model, _EvalLoader(ds, 128), ev, 'cuda')
            for k, v in fresh.items():
                assert best[j][k] == v, (j, k, best[j][k], v)
            assert best[j]['max_optimizing_metric'] == best[j]['ndcg@10']
