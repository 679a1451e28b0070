"""GPU: packed validation — hsk_eval_topk_pack bitwise against hsk_eval_topk per trial (random tables, one per trial) and
against the float64 reference on exact-score tables (tests/topk_exact.py), hsk_rank_metrics_pack and
hsk_rank_metrics_sums_det_pack against their single-model kernels, evaluate_mf_pack against
evaluate_recommender_algorithm per trial, guard words, status bits, and PackedTrainer's per-trial fallback for tensor-core
evaluation."""
import os
import tempfile

import numpy as np
import pytest
import torch

import topk_exact as X

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def _pack_models(M, U, I, d, biases, seed0=0):
    """M SGDMatrixFactorization models, each with its own random tables, bound to the rows of one [M, stride] allocation
    (as PackedMFTrainStep binds them).  Returns (models, p)."""
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    models = []
    for j in range(M):
        m = SGDMatrixFactorization.on_device(U, I, d, *biases, device='cuda', seed=seed0 + 31 * j, std=(d ** -0.5, 0.05))
        if biases[2]:
            m.global_bias.data.fill_(0.01 * (j + 1))
        models.append(m)
    p = torch.empty((M, models[0].layout.n_total), dtype=torch.float32, device='cuda')
    for j, m in enumerate(models):
        p[j].copy_(m.arena.detach())
        m._set_arena(p[j])
    return models, p


def _exclusions(kind, U, I, seed=0):
    """None, or the (indptr, indices) device CSR of one exclusion row per user: 'rand' = 0..40 random items (some rows
    empty); 'tail' = 'rand' plus every 50th user keeps only 3 admissible items (fewer than k: the -inf tail)."""
    if kind == 'none':
        return None, None
    rng = np.random.RandomState(seed)
    rows = []
    for u in range(U):
        if kind == 'tail' and u % 50 == 0:
            rows.append(np.setdiff1d(np.arange(I), rng.choice(I, min(I, 3), replace=False)).astype(np.int32))
        else:
            rows.append(np.unique(rng.randint(0, I, rng.randint(0, min(I, 40) + 1))).astype(np.int32))
    indptr, indices = X.csr(rows)
    if len(indices) == 0:
        indices = np.zeros(1, np.int32)
    return torch.from_numpy(indptr).cuda(), torch.from_numpy(indices).cuda()


def _users(U, Be, seed=0):
    """A batch with repeated users."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randint(0, U, (Be,), generator=g)
    if Be > 1:
        u[Be - 1] = u[0]
    return u.cuda()


def _single(model, u, k, ex_p, ex_i):
    from hassaku_b200 import _C
    Be = u.numel()
    s = torch.empty((Be, k), dtype=torch.float32, device='cuda')
    i = torch.empty((Be, k), dtype=torch.int32, device='cuda')
    scratch = torch.empty(_C.eval_topk_scratch_bytes(Be, model.n_items, k), dtype=torch.uint8, device='cuda')
    _C.eval_topk(model._tables(), u, k, s, i, scratch, ex_p, ex_i)
    return s, i


def _packed(models, p, active_idx, u, k, ex_p, ex_i, status=None):
    from hassaku_b200 import _C
    A, Be = len(active_idx), u.numel()
    active = torch.tensor(active_idx, dtype=torch.int32, device='cuda')
    s = torch.empty((A, Be, k), dtype=torch.float32, device='cuda')
    i = torch.empty((A, Be, k), dtype=torch.int32, device='cuda')
    scratch = torch.empty(_C.eval_topk_pack_scratch_bytes(Be, models[0].n_items, k, A), dtype=torch.uint8, device='cuda')
    _C.eval_topk_pack(models[0].layout.tables(p[0]), p.shape[1], p.shape[0], active, u, k, s, i, scratch, ex_p, ex_i,
                      status=status)
    return s, i


# (d, items, Be, k, biases, M, active): every d, catalogue, batch and k of the grid, several splits at 250 k items,
# non-contiguous and reversed active subsets
NONE, ALL = (False, False, False), (True, True, True)
TOPK_CASES = [
    (7, 1, 1, 1, NONE, 1, [0]),
    (64, 100, 64, 100, ALL, 3, [2, 0]),
    (402, 3706, 1000, 100, ALL, 17, [16, 13, 9, 4, 1]),
    (1024, 3706, 64, 128, NONE, 3, [1, 2]),
    (64, 250_000, 1, 100, ALL, 3, [2, 0, 1]),
    (7, 250_000, 64, 128, NONE, 17, [15, 3, 8]),
    (402, 100, 8192, 1, ALL, 3, [0, 2]),
    (64, 3706, 8192, 100, ALL, 17, list(range(16, -1, -2))),
    (1024, 250_000, 1000, 100, ALL, 3, [1]),
    (7, 100, 1000, 128, ALL, 1, [0]),
]


@pytest.mark.parametrize('excl', ['none', 'rand', 'tail'])
@pytest.mark.parametrize('d,I,Be,k,biases,M,active', TOPK_CASES)
def test_eval_topk_pack_bitwise_vs_single_model(d, I, Be, k, biases, M, active, excl):
    U = 1500
    models, p = _pack_models(M, U, I, d, biases)
    ex_p, ex_i = _exclusions(excl, U, I)
    u = _users(U, Be)
    s, i = _packed(models, p, active, u, k, ex_p, ex_i)
    for a, j in enumerate(active):
        ws, wi = _single(models[j], u, k, ex_p, ex_i)
        assert torch.equal(i[a], wi), (j, int((i[a] != wi).sum()))
        assert torch.equal(_bits(s[a]), _bits(ws)), j


@pytest.mark.parametrize('I', [1000, 70_000])
@pytest.mark.parametrize('k', [1, 100, 128])
def test_eval_topk_pack_exact_tables(I, k):
    """Each trial of the pack holds a different exact-score table (digit orders with integer biases, digit orders with an
    item bias, one 16-bit key prefix per item — digit orders without biases above the prefix table's 32 000 items —, +0 /
    -0 ties): ids and scores equal the float64 reference bitwise (+0 and -0 count as one score)."""
    from hassaku_b200 import _C
    from hassaku_b200.algorithms.sgd_alg import ArenaLayout
    d = 32
    orders = list(X.ORDERS)
    U = len(orders)
    tabs = [X.make_tables('digits', I, d, orders, 'all', seed=0),
            X.make_tables('digits', I, d, orders[::-1], 'ib', seed=1),
            X.make_tables('prefix', I, d, orders) if I <= 32000
            else X.make_tables('digits', I, d, orders[3:] + orders[:3], seed=3),
            X.make_tables('zeros', I, d, orders, seed=2)]
    M = len(tabs)
    for t in tabs:   # one pack shape: every trial has user, item and global biases (0 where its table has none)
        t.Ub = np.zeros(U, np.float32) if t.Ub is None else t.Ub
        t.Gb = np.zeros(1, np.float32) if t.Gb is None else t.Gb
        t.Ib = np.zeros(I, np.float32) if t.Ib is None else t.Ib
    lay = ArenaLayout(U, I, d, True, True, True)
    p = torch.zeros((M, lay.n_total), dtype=torch.float32, device='cuda')
    for j, t in enumerate(tabs):
        Uw, Vw, Ub, Ib, Gb = lay.views(p[j])
        for dst, src in ((Uw, t.Uw), (Vw, t.Vw), (Ub, t.Ub[:, None]), (Ib, t.Ib[:, None]), (Gb, t.Gb)):
            dst.copy_(torch.from_numpy(np.ascontiguousarray(src).reshape(dst.shape)))
    ex_rows = [X.exclusions(kind, tabs[0].scores()[u], seed=u)
               for u, kind in zip(range(U), ['none', 'rand', 'top', 'edges', 'allbut3', 'all'] * U)]
    indptr, indices = X.csr(ex_rows)
    ex_p, ex_i = torch.from_numpy(indptr).cuda(), torch.from_numpy(indices).cuda()
    u_np = np.concatenate([np.arange(U), np.arange(U)[::-1], [U]])    # repeated users and one invalid index
    u = torch.from_numpy(u_np).cuda()
    active = [3, 1, 2, 0]
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    act = torch.tensor(active, dtype=torch.int32, device='cuda')
    s = torch.empty((M, len(u_np), k), dtype=torch.float32, device='cuda')
    i = torch.empty((M, len(u_np), k), dtype=torch.int32, device='cuda')
    scratch = torch.empty(_C.eval_topk_pack_scratch_bytes(len(u_np), I, k, M), dtype=torch.uint8, device='cuda')
    _C.eval_topk_pack(lay.tables(p[0]), lay.n_total, M, act, u, k, s, i, scratch, ex_p, ex_i, status=status)
    assert int(status.item()) & _C.STATUS_BAD_INDEX
    for a, j in enumerate(active):
        want_i, want_s = X.expand_rows(*X.reference_topk(tabs[j].scores(), ex_rows, k), u_np, U)
        assert np.array_equal(i[a].cpu().numpy(), want_i), j
        assert np.array_equal(s[a].cpu().numpy(), want_s), j     # == : bitwise up to the sign of zero


def _labels(U, I, seed=0):
    rng = np.random.RandomState(seed)
    rows = [np.unique(rng.randint(0, I, rng.randint(0, 30))).astype(np.int32) for _ in range(U)]
    indptr, indices = X.csr(rows)
    return torch.from_numpy(indptr).cuda(), torch.from_numpy(indices).cuda()


def _metric_inputs(M, Be, U, I, k_max, G, seed=0):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(-1, I, (M, Be, k_max), generator=g, dtype=torch.int32).cuda()
    u = torch.randint(0, U, (Be,), generator=g).cuda()
    grp = torch.randint(0, max(G, 1), (U,), generator=g, dtype=torch.int32).cuda() if G else None
    return ids, u, grp


KS = [100, 50, 10, 5]


@pytest.mark.parametrize('G', [0, 2, 5])
@pytest.mark.parametrize('Be', [1, 64, 1000])
def test_rank_metrics_pack_vs_single_model(G, Be):
    """per_user bitwise, sums up to fp64 reordering, counts exact; inactive trials' sums / counts untouched."""
    from hassaku_b200 import _C
    from hassaku_b200.eval.metrics import discount_table
    U, I, T, active = 400, 300, 5, [4, 1, 2]
    lab_p, lab_i = _labels(U, I)
    ids, u, grp = _metric_inputs(len(active), Be, U, I, KS[0], G)
    disc = discount_table(KS[0], 'cuda')
    sums = torch.full((T, 1 + G, len(KS), 3), 0.25, dtype=torch.float64, device='cuda')
    counts = torch.full((T, 1 + G), 3, dtype=torch.int64, device='cuda')
    per_user = torch.empty((len(active), Be, len(KS), 3), dtype=torch.float32, device='cuda')
    act = torch.tensor(active, dtype=torch.int32, device='cuda')
    _C.rank_metrics_pack(ids, KS, u, lab_p, lab_i, disc, act, sums, counts, user_group=grp, n_groups=G, per_user=per_user)
    for j in set(range(T)) - set(active):
        assert float(sums[j].min()) == 0.25 and float(sums[j].max()) == 0.25 and int(counts[j].min()) == 3
        assert int(counts[j].max()) == 3
    for a, j in enumerate(active):
        ws = torch.full((1 + G, len(KS), 3), 0.25, dtype=torch.float64, device='cuda')
        wc = torch.full((1 + G,), 3, dtype=torch.int64, device='cuda')
        wp = torch.empty((Be, len(KS), 3), dtype=torch.float32, device='cuda')
        _C.rank_metrics(ids[a].contiguous(), KS, u, lab_p, lab_i, disc, ws, wc, user_group=grp, n_groups=G, per_user=wp)
        assert torch.equal(_bits(per_user[a]), _bits(wp)), j
        assert torch.equal(counts[j], wc), j
        torch.testing.assert_close(sums[j], ws, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('G', [0, 2, 5])
@pytest.mark.parametrize('batch', [1, 64, 128])
def test_rank_metrics_sums_det_pack_bitwise_per_batch(G, batch):
    """Chunks of several batches (the last one short): bitwise what one hsk_rank_metrics_sums_det call per batch gives,
    in order, from non-zero starting sums; inactive trials untouched."""
    from hassaku_b200 import _C
    U, T, active = 400, 4, [3, 0]
    Be = 5 * batch - (batch // 2)
    g = torch.Generator().manual_seed(batch + G)
    per_user = (torch.rand((len(active), Be, len(KS), 3), generator=g) * torch.rand(1, generator=g)).cuda()
    u = torch.randint(0, U, (Be,), generator=g).cuda()
    grp = torch.randint(0, G, (U,), generator=g, dtype=torch.int32).cuda() if G else None
    start = torch.rand((T, 1 + G, len(KS), 3), generator=g, dtype=torch.float64).cuda()
    sums = start.clone()
    act = torch.tensor(active, dtype=torch.int32, device='cuda')
    _C.rank_metrics_sums_det_pack(per_user, u, batch, act, sums, user_group=grp, n_groups=G)
    assert torch.equal(sums[1], start[1]) and torch.equal(sums[2], start[2])
    for a, j in enumerate(active):
        want = start[j].clone()
        for b0 in range(0, Be, batch):
            _C.rank_metrics_sums_det(per_user[a, b0:b0 + batch].contiguous(), u[b0:b0 + batch].contiguous(), want,
                                     user_group=grp, n_groups=G)
        assert torch.equal(_bits(sums[j].view(torch.float32)), _bits(want.view(torch.float32))), j


# ---------------------------------------------------------------------------------------------------------------------
# evaluate_mf_pack
# ---------------------------------------------------------------------------------------------------------------------
class _EvalLoader:
    def __init__(self, dataset, batch_size):
        self.dataset, self.batch_size = dataset, batch_size


def _val_dataset(U=700, I=300, G=2, seed=0):
    from hassaku_b200.data.dataset import FullEvalDataset
    from hassaku_b200.data.synthetic import make_interactions
    data = make_interactions(U, I, 14 * U, seed=seed, n_user_groups=G)
    return FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, G)


@pytest.fixture
def det_mode():
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    yield lambda: torch.use_deterministic_algorithms(True)
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


@pytest.mark.parametrize('deterministic', [False, True])
@pytest.mark.parametrize('bs', [64, 128, 'all'])
@pytest.mark.parametrize('budget', ['default', 'small'])
def test_evaluate_mf_pack_equals_per_trial(bs, deterministic, budget, det_mode, monkeypatch):
    """Entries equal evaluate_recommender_algorithm per trial (== in default mode, bitwise under determinism) for a
    reversed, non-contiguous subset of the pack; the small scratch budget makes chunks of three loader batches."""
    from hassaku_b200.eval import eval as E
    ds = _val_dataset()
    bs = ds.n_users if bs == 'all' else bs
    models, _p = _pack_models(5, ds.n_users, ds.n_items, 48, ALL, seed0=3)
    trials = [4, 1, 2]
    if budget == 'small':
        monkeypatch.setattr(E, 'PACK_SCRATCH_BYTES', 3 * bs * len(trials) * E._C.eval_topk_pack_scratch_bytes(1, ds.n_items, 100, 1))
        assert E.pack_chunk_users(bs, ds.n_users, ds.n_items, 100, len(trials), E.PACK_SCRATCH_BYTES) == min(
            3 * bs, -(-ds.n_users // bs) * bs)
    if deterministic:
        det_mode()
    mk = lambda: E.FullEvaluator(aggr_by_group=True, n_groups=ds.n_user_groups, user_to_user_group=ds.user_to_user_group)
    got = E.evaluate_mf_pack([models[j] for j in trials], _EvalLoader(ds, bs), [mk() for _ in trials], 'cuda')
    for a, j in enumerate(trials):
        want = E.evaluate_recommender_algorithm(models[j], _EvalLoader(ds, bs), mk(), 'cuda')
        assert got[a].keys() == want.keys()
        for key in want:
            assert got[a][key] == want[key], (j, key, got[a][key], want[key])
            if deterministic:
                assert np.float64(got[a][key]).tobytes() == np.float64(want[key]).tobytes(), (j, key)


def test_evaluate_mf_pack_raises_on_out_of_range_user():
    """Models with fewer users than the dataset: the packed sweep raises IndexError, as the per-model sweep does."""
    from hassaku_b200.eval import eval as E
    ds = _val_dataset(U=300)
    models, _p = _pack_models(2, 250, ds.n_items, 16, NONE)
    mk = lambda: E.FullEvaluator(aggr_by_group=True, n_groups=ds.n_user_groups, user_to_user_group=ds.user_to_user_group)
    with pytest.raises(IndexError):
        E.evaluate_recommender_algorithm(models[0], _EvalLoader(ds, 64), mk(), 'cuda')
    with pytest.raises(IndexError):
        E.evaluate_mf_pack(models, _EvalLoader(ds, 64), [mk(), mk()], 'cuda')


def test_pack_status_bits():
    """An out-of-range active entry and an out-of-range user set HSK_STATUS_BAD_INDEX; the bad user's rows are -1 / -inf
    and the other rows are the single-model kernel's."""
    from hassaku_b200 import _C
    U, I, k = 200, 500, 100
    models, p = _pack_models(3, U, I, 16, ALL)
    u = _users(U, 64)
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    _packed(models, p, [0, 3], u, k, None, None, status=status)
    assert int(status.item()) & _C.STATUS_BAD_INDEX
    status.zero_()
    u_bad = u.clone(); u_bad[5] = U
    s, i = _packed(models, p, [2, 0], u_bad, k, None, None, status=status)
    assert int(status.item()) & _C.STATUS_BAD_INDEX
    assert bool((i[:, 5] == -1).all()) and bool(torch.isinf(s[:, 5]).all())
    ws, wi = _single(models[2], u, k, None, None)
    keep = torch.arange(64, device='cuda') != 5
    assert torch.equal(i[0][keep], wi[keep])
    status.zero_()
    sums = torch.zeros((3, 1, len(KS), 3), dtype=torch.float64, device='cuda')
    counts = torch.zeros((3, 1), dtype=torch.int64, device='cuda')
    from hassaku_b200.eval.metrics import discount_table
    lab_p, lab_i = _labels(U, I)
    _C.rank_metrics_pack(wi[None].contiguous(), KS, u, lab_p, lab_i, discount_table(100, 'cuda'),
                         torch.tensor([3], dtype=torch.int32, device='cuda'), sums, counts, status=status)
    assert int(status.item()) & _C.STATUS_BAD_INDEX and int(counts.abs().sum()) == 0
    status.zero_()
    per_user = torch.rand((1, 64, len(KS), 3), device='cuda')
    _C.rank_metrics_sums_det_pack(per_user, u, 64, torch.tensor([-1], dtype=torch.int32, device='cuda'), sums, status=status)
    assert int(status.item()) & _C.STATUS_BAD_INDEX and float(sums.abs().sum()) == 0.0


class _Guarded:
    """A tensor carved out of a larger allocation whose margins hold a canary pattern (as test_gpu_trial_pack.py's)."""
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


@pytest.mark.parametrize('I', [3706, 250_000])
def test_pack_kernels_do_not_write_outside_their_buffers(I):
    from hassaku_b200 import _C
    from hassaku_b200.eval.metrics import discount_table
    U, Be, k, T, G, active = 900, 300, 100, 4, 2, [3, 1]
    A = len(active)
    models, p = _pack_models(T, U, I, 64, ALL)
    ex_p, ex_i = _exclusions('tail', U, I)
    u = _users(U, Be)
    act = _Guarded((A,), torch.int32)
    act.t.copy_(torch.tensor(active, dtype=torch.int32))
    s, i = _Guarded((A, Be, k), torch.float32), _Guarded((A, Be, k), torch.int32)
    scratch = _Guarded((_C.eval_topk_pack_scratch_bytes(Be, I, k, A),), torch.uint8)
    status = _Guarded((1,), torch.int32, 0)
    _C.eval_topk_pack(models[0].layout.tables(p[0]), p.shape[1], T, act.t, u, k, s.t, i.t, scratch.t, ex_p, ex_i,
                      status=status.t)
    sums = _Guarded((T, 1 + G, len(KS), 3), torch.float64, 0.0)
    counts = _Guarded((T, 1 + G), torch.int64, 0)
    per_user = _Guarded((A, Be, len(KS), 3), torch.float32)
    lab_p, lab_i = _labels(U, I)
    grp = torch.randint(0, G, (U,), dtype=torch.int32, device='cuda')
    _C.rank_metrics_pack(i.t, KS, u, lab_p, lab_i, discount_table(k, 'cuda'), act.t, sums.t, counts.t, user_group=grp,
                         n_groups=G, per_user=per_user.t, status=status.t)
    _C.rank_metrics_sums_det_pack(per_user.t, u, 64, act.t, sums.t, user_group=grp, n_groups=G, status=status.t)
    torch.cuda.synchronize()
    assert int(status.t.item()) == 0
    for x in (act, s, i, scratch, status, sums, counts, per_user):
        assert x.intact()
    for j in (0, 2):    # inactive trials
        assert float(sums.t[j].abs().sum()) == 0.0 and int(counts.t[j].abs().sum()) == 0


# ---------------------------------------------------------------------------------------------------------------------
# PackedTrainer: per-trial fallback for tensor-core evaluation
# ---------------------------------------------------------------------------------------------------------------------
def test_packed_trainer_bf16_eval_falls_back_to_per_trial_val(det_mode):
    from hassaku_b200.data.dataloader import NegativeSampler, TrainDataLoader
    from hassaku_b200.data.dataset import FullEvalDataset, TrainRecDataset
    from hassaku_b200.data.synthetic import make_interactions
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer import Trainer
    from hassaku_b200.train.trial_pack import PackedTrainer
    data = make_interactions(300, 200, 6000, seed=0, n_user_groups=2)
    tds = TrainRecDataset.from_interactions(data.train, data.user_group, 2)
    ds = FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, 2)
    loader = lambda: TrainDataLoader(NegativeSampler(tds, n_neg=20), tds, batch_size=256, shuffle=True, seed=7)
    trials = [dict(seed=1, lr=5e-3, wd=1e-5, n_epochs=2, max_patience=5), dict(seed=2, lr=0.0, wd=1e-4, n_epochs=3, max_patience=1)]

    def model(seed):
        torch.manual_seed(seed)
        m = SGDMatrixFactorization(300, 200, 32, use_item_bias=True)
        with torch.no_grad():
            m.user_embeddings.weight.mul_(40.)
            m.item_embeddings.weight.mul_(40.)
        m.eval_precision = 'bf16'
        return m

    def conf(t, path):
        return {'device': 'cuda', 'lr': t['lr'], 'wd': t['wd'], 'optimizer': 'adamw', 'n_epochs': t['n_epochs'],
                'optimizing_metric': 'ndcg@10', 'max_patience': t['max_patience'], 'model_path': path,
                'running_settings': {'use_wandb': False, 'batch_verbose': False}}

    det_mode()
    with tempfile.TemporaryDirectory() as tmp:
        paths = [os.path.join(tmp, f'pack{j}') for j in range(len(trials))]
        for pth in paths:
            os.makedirs(pth)
        pt = PackedTrainer([model(t['seed']) for t in trials], loader(), _EvalLoader(ds, 128),
                           RecBayesianPersonalizedRankingLoss(), [conf(t, pth) for t, pth in zip(trials, paths)])
        assert pt.val_pack([0, 1]) == {}
        got = pt.fit()
        for j, t in enumerate(trials):
            pth = os.path.join(tmp, f'single{j}')
            os.makedirs(pth)
            want = Trainer(model(t['seed']), loader(), _EvalLoader(ds, 128), RecBayesianPersonalizedRankingLoss(),
                           conf(t, pth)).fit()
            assert got[j] == want, j
