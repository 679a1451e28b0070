"""GPU: the deterministic mode (torch.use_deterministic_algorithms(True)) — the gradient scatter bit-exact against the
numpy restatement of its order contract (oracle/det_oracle.py), the fused deterministic step against the reference math,
bitwise reproducible steps and training runs, and the sharded step's refusal."""
import math
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-5


@pytest.fixture
def det_mode():
    """Call it to turn torch.use_deterministic_algorithms on (after building data: data/synthetic.py's CUDA cumsum has no
    deterministic implementation); the previous state, warn_only included, is restored afterwards."""
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())

    def enable(warn_only=False):
        torch.use_deterministic_algorithms(True, warn_only=warn_only)

    yield enable
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def bits_equal(got, want):
    np.testing.assert_array_equal(np.ascontiguousarray(got, np.float32).view(np.int32),
                                  np.ascontiguousarray(want, np.float32).view(np.int32))


def make_model(U, I, d, biases, seed=1):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    torch.manual_seed(seed)
    m = SGDMatrixFactorization(U, I, d, *biases)
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn_like(p) * (1.0 / math.sqrt(d) if p.shape[-1] == d else 0.1))
    return m.to('cuda')


def make_batch(rng, U, I, B, N, head_share=0.0):
    """Zipf-skewed positives, repeated users; head_share of the positives on item 7."""
    p = 1. / np.arange(1, I + 1) ** 0.8
    p /= p.sum()
    u = rng.randint(0, U, B).astype(np.int64)
    u[:B // 8] = u[0]
    pos = rng.choice(I, B, p=p)
    pos[rng.rand(B) < head_share] = 7
    i = np.column_stack([pos, rng.randint(0, I, (B, N))]).astype(np.int64)
    return u, i


def grads_np(model, g_arena):
    names = ('gU', 'gV', 'gUb', 'gIb', 'gGb')
    return {n: None if v is None else v.detach().cpu().numpy() for n, v in zip(names, model.layout.views(g_arena))}


def check_against_oracle(model, g_arena, u, i, ds):
    from oracle import det_oracle as D
    Uw = model.user_embeddings.weight.detach().cpu().numpy()
    Vw = model.item_embeddings.weight.detach().cpu().numpy()
    want = D.scatter_grads(Uw, Vw, u, i, ds, (model.use_user_bias, model.use_item_bias, model.use_global_bias))
    got = grads_np(model, g_arena)
    for k, w in want.items():
        if w is None:
            assert got[k] is None
            continue
        bits_equal(got[k].reshape(w.shape), w)


SCATTER = [
    # U, I, d, B, N, biases (u, i, g), head share of the positives
    (300, 200, 7, 64, 5, (True, True, True), 0.0),
    (2000, 1500, 128, 512, 20, (False, True, False), 0.0),
    (2000, 1500, 128, 512, 20, (False, False, False), 0.0),
    (1000, 800, 402, 256, 10, (True, True, True), 0.0),
    (300, 500, 1024, 33, 4, (False, False, True), 0.0),
    (1000, 2000, 64, 2048, 10, (True, True, False), 0.4),      # item 7 owns > 30 % of the positives: many chunks
    (6040, 3706, 402, 8192, 50, (False, True, False), 0.0),    # cfg2 batch shape
]


@pytest.mark.parametrize('U,I,d,B,N,biases,head', SCATTER)
def test_scatter_bit_exact_vs_order_oracle(U, I, d, B, N, biases, head):
    from hassaku_b200 import _C
    model = make_model(U, I, d, biases)
    rng = np.random.RandomState(5)
    u, i = make_batch(rng, U, I, B, N, head)
    ds = (rng.randn(B, N + 1) * 1e-3).astype(np.float32)
    ut, it, dst = torch.from_numpy(u).cuda(), torch.from_numpy(i).cuda(), torch.from_numpy(ds).cuda()
    lay = model.layout
    scratch = torch.empty(_C.det_scratch_bytes(B, N + 1, lay.ld), dtype=torch.uint8, device='cuda')
    runs = []
    for _ in range(2):
        g = torch.zeros(lay.n_total, dtype=torch.float32, device='cuda')
        _C.mf_scatter_grads_det(model._tables(), lay.tables(g), ut, it, dst, scratch, model._status())
        runs.append(g)
    assert torch.equal(runs[0], runs[1])
    model.check_status()
    check_against_oracle(model, runs[0], u, i, ds)
    if lay.ld != d:   # pad columns stay zero
        assert float(runs[0][:U * lay.ld].view(U, lay.ld)[:, d:].abs().max()) == 0.0


FUSED = [
    ('bpr', (False, True, False), 128), ('bpr', (True, False, True), 402), ('bpr', (True, True, True), 7),
    ('sampled_softmax', (False, True, False), 128), ('sampled_softmax', (True, True, True), 402),
    ('sampled_softmax', (False, False, False), 64),
    ('bce', (True, True, True), 128), ('bce', (False, False, False), 402), ('bce', (False, True, False), 1024),
]


def loss_fn(kind, I, N):
    from hassaku_b200.train.rec_losses import RecommenderSystemLossesEnum

    class _DS:
        n_items = I

    return RecommenderSystemLossesEnum[kind].value.build_from_conf({'train_neg_strategy': 'uniform', 'neg_train': N}, _DS())


@pytest.mark.parametrize('kind,biases,d', FUSED)
def test_fused_det_step_vs_reference_math(kind, biases, d, det_mode):
    """Scores, loss and dL/ds at the tolerances of test_gpu_train.py's fused-step gate; gradients bitwise equal to the order
    oracle applied to the step's own dL/ds; one teacher-forced AdamW step within the per-step gate of the default step."""
    from oracle import mf_oracle as O
    from hassaku_b200 import _C
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    U, I, B, N = 2000, 1500, 256, 20
    model = make_model(U, I, d, biases)
    rng = np.random.RandomState(2)
    u, i = make_batch(rng, U, I, B, N)
    ut, it = torch.from_numpy(u).cuda(), torch.from_numpy(i).cuda()
    ref = O.OracleMF(U, I, d, *biases)
    ref.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()})
    r = O.OracleTrainer(ref, kind, 1e-3, 1e-2, 'adamw', neg_train=N).step(torch.from_numpy(u), torch.from_numpy(i), keep=True)
    lay = model.layout
    loss_fn_ = loss_fn(kind, I, N)
    g = torch.zeros(lay.n_total, dtype=torch.float32, device='cuda')
    loss = torch.zeros(1, dtype=torch.float64, device='cuda')
    scores = torch.empty((B, N + 1), dtype=torch.float32, device='cuda')
    dsc = torch.empty((B, N + 1), dtype=torch.float32, device='cuda')
    scratch = torch.empty(_C.det_scratch_bytes(B, N + 1, lay.ld), dtype=torch.uint8, device='cuda')
    _C.mf_train_fused_det(model._tables(), lay.tables(g), ut, it, _C.LOSS_KINDS[kind], loss_fn_.neg_shift(), loss, scratch,
                          scores_out=scores, dscores_out=dsc, status=model._status())
    model.check_status()
    assert rel_err(scores.cpu().numpy(), r['scores'].numpy()) < RTOL
    assert rel_err(dsc.cpu().numpy(), r['dscores'].numpy()) < RTOL
    assert abs(float(loss) - float(r['loss'])) <= RTOL * abs(float(r['loss']))
    check_against_oracle(model, g, u, i, dsc.cpu().numpy())

    # one step through FusedMFTrainStep under the switch vs the default step from the same state
    sd0 = {k: v.clone() for k, v in model.state_dict().items()}
    params = []
    for det in (False, True):
        model.load_state_dict(sd0)
        opt = DenseAdam(model, lr=1e-3, weight_decay=1e-2)
        step = FusedMFTrainStep(model, loss_fn_, opt)
        if det:
            det_mode()
        step(ut, it)
        step.pop_loss_sum()
        params.append({n: p.detach().cpu().numpy().copy() for n, p in model.named_parameters()})
    lr = 1e-3
    for n, want in params[0].items():
        if kind in ('bpr', 'sampled_softmax') and n in ('user_bias.weight', 'global_bias'):
            continue   # invariant directions: only Adam's |dp| <= lr bound is checkable (test_gpu_train.py)
        err = np.abs(params[1][n].astype(np.float64) - want).max()
        assert err < RTOL * np.abs(want).max() + 2e-3 * lr, (n, err)


def _run_steps(model, arena0, batches):
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    with torch.no_grad():
        model.arena.copy_(arena0)
    opt = DenseAdam(model, lr=1e-3, weight_decay=1e-2)
    step = FusedMFTrainStep(model, RecBayesianPersonalizedRankingLoss(), opt)
    losses = []
    for u, i in batches:
        step(u, i)
        losses.append(step.pop_loss_sum())
    return [model.arena.clone(), opt.m.clone(), opt.v.clone()], losses


REPRO = [
    # U, I, d, B, N, steps
    (2000, 1500, 128, 512, 50, 5),
    (6040, 3706, 402, 8192, 50, 5),               # cfg2 shape
    (2_000_000, 1_000_000, 128, 8192, 50, 2),     # cfg4 shape
]


@pytest.mark.parametrize('U,I,d,B,N,steps', REPRO)
def test_steps_bitwise_reproducible(U, I, d, B, N, steps, det_mode):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    model = SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=3)
    arena0 = model.arena.clone()
    gen = torch.Generator(device='cuda')
    gen.manual_seed(11)
    batches = [(torch.randint(0, U, (B,), device='cuda', generator=gen),
                torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)) for _ in range(steps)]
    det_mode()
    a, la = _run_steps(model, arena0, batches)
    b, lb = _run_steps(model, arena0, batches)
    assert la == lb
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize('kind', ['bpr', 'sampled_softmax', 'bce'])
def test_autograd_path_bitwise_and_vs_order_oracle(kind, det_mode):
    from oracle import mf_oracle as O
    U, I, d, B, N = 1500, 900, 64, 384, 12
    biases = (True, True, True)
    model = make_model(U, I, d, biases)
    rng = np.random.RandomState(4)
    u, i = make_batch(rng, U, I, B, N, 0.3)
    labels = O.make_labels(B, N + 1).cuda()
    det_mode()
    runs = []
    for _ in range(2):
        model.zero_grad()
        out = model(torch.from_numpy(u).cuda(), torch.from_numpy(i).cuda())
        cap = {}
        out.register_hook(lambda gr: cap.__setitem__('g', gr.detach().clone()))
        loss = loss_fn(kind, I, N).compute_loss(out, labels)
        loss.backward()
        runs.append((loss.detach().clone(), cap['g'], {n: p.grad.clone() for n, p in model.named_parameters()}))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for n in runs[0][2]:
        assert torch.equal(runs[0][2][n], runs[1][2][n]), n
    from oracle import det_oracle as D
    ds = runs[0][1].cpu().numpy()
    want = D.scatter_grads(model.user_embeddings.weight.detach().cpu().numpy(),
                           model.item_embeddings.weight.detach().cpu().numpy(), u, i, ds, biases)
    got = {n: g.cpu().numpy() for n, g in runs[0][2].items()}
    bits_equal(got['user_embeddings.weight'], want['gU'])
    bits_equal(got['item_embeddings.weight'], want['gV'])
    bits_equal(got['user_bias.weight'].ravel(), want['gUb'])
    bits_equal(got['item_bias.weight'].ravel(), want['gIb'])
    bits_equal(got['global_bias'], want['gGb'])


class _EvalLoader:
    def __init__(self, dataset, batch_size):
        self.dataset, self.batch_size = dataset, batch_size


@pytest.mark.parametrize('optimizer,mode', [('adamw', 'dense'), ('adam', 'dense'), ('adagrad', 'dense'), ('adamw', 'lazy')])
def test_trainer_fit_twice_identical(optimizer, mode, det_mode):
    """Trainer.fit() twice under the switch with the device loader and a user group: identical checkpoints, metric dicts
    and epoch losses."""
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.data.dataloader import NegativeSampler, TrainDataLoader
    from hassaku_b200.data.dataset import FullEvalDataset, TrainRecDataset
    from hassaku_b200.data.synthetic import make_interactions
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer import Trainer
    data = make_interactions(300, 200, 6000, seed=0, n_user_groups=2)
    tds = TrainRecDataset.from_interactions(data.train, data.user_group, 2)
    ds = FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, 2)
    det_mode()
    results = []
    for _ in range(2):
        dl = TrainDataLoader(NegativeSampler(tds, n_neg=20), tds, batch_size=256, shuffle=True, seed=7)
        torch.manual_seed(1)
        model = SGDMatrixFactorization(300, 200, 32, use_item_bias=True)
        with torch.no_grad():
            model.user_embeddings.weight.mul_(40.)
            model.item_embeddings.weight.mul_(40.)
        conf = {'device': 'cuda', 'lr': 5e-3, 'wd': 1e-5, 'optimizer': optimizer, 'optimizer_mode': mode, 'n_epochs': 2,
                'optimizing_metric': 'ndcg@10', 'max_patience': 5,
                'running_settings': {'use_wandb': False, 'batch_verbose': False}}
        with tempfile.TemporaryDirectory() as tmp:
            conf['model_path'] = tmp
            tr = Trainer(model, dl, _EvalLoader(ds, 128), RecBayesianPersonalizedRankingLoss(), conf)
            logs = []
            tr._report = lambda log_dict, epoch: logs.append(dict(log_dict))
            best = tr.fit()
            sd = torch.load(os.path.join(tmp, 'model.pth'), map_location='cpu')
        results.append((best, logs, sd))
    (b0, l0, s0), (b1, l1, s1) = results
    assert b0 == b1
    assert l0 == l1 and len(l0) == 3
    assert [x['epoch_train_loss'] for x in l0[1:]] == [x['epoch_train_loss'] for x in l1[1:]]
    assert len([k for k in b0 if k.startswith('group_')]) == 24
    assert set(s0) == set(s1)
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k


def test_eval_sums_fixed_order_per_group(det_mode):
    """FullEvaluator under the switch: the per-group sums are the fixed-order sums of the per-user values."""
    from hassaku_b200.eval.eval import FullEvaluator
    rng = np.random.RandomState(0)
    Be, I, n_groups = 3000, 500, 3
    logits = torch.from_numpy(rng.randn(Be, I).astype(np.float32)).cuda()
    y = torch.from_numpy((rng.rand(Be, I) < 0.05).astype(np.float32)).cuda()
    u = torch.arange(Be, device='cuda')
    grp = torch.from_numpy(rng.randint(0, n_groups, Be).astype(np.int32))
    det_mode()
    res = []
    for _ in range(2):
        ev = FullEvaluator(aggr_by_group=True, n_groups=n_groups, user_to_user_group=grp)
        ev.eval_batch(u[:1700], logits[:1700], y[:1700])
        ev.eval_batch(u[1700:], logits[1700:], y[1700:])
        res.append(ev.get_results())
    assert res[0] == res[1]
    torch.use_deterministic_algorithms(False)
    ev = FullEvaluator(aggr_by_group=True, n_groups=n_groups, user_to_user_group=grp)
    ev.eval_batch(u, logits, y)
    ref = ev.get_results()
    assert set(ref) == set(res[0])
    for k, v in ref.items():
        assert abs(res[0][k] - v) <= 1e-12 + 1e-12 * abs(v), k


def test_sharded_step_raises_or_warns_under_the_switch(det_mode):
    from hassaku_b200.sharded import ShardedMF
    U, I, d, B, N = 200, 150, 16, 32, 4
    smf = ShardedMF(U, I, d, use_item_bias=True, world=1, rank=0, device='cuda')
    u = torch.randint(0, U, (B,), device='cuda')
    i = torch.randint(0, I, (B, N + 1), device='cuda')
    det_mode()
    with pytest.raises(RuntimeError, match='deterministic'):
        smf.step(u, i, B, 'bpr', 0.0, 1e-3, 0.0, exchange='sparse')
    det_mode(warn_only=True)
    with pytest.warns(UserWarning, match='deterministic'):
        smf.step(u, i, B, 'bpr', 0.0, 1e-3, 0.0, exchange='sparse')
    torch.use_deterministic_algorithms(False)
    smf.step(u, i, B, 'bpr', 0.0, 1e-3, 0.0, exchange='sparse')
    assert math.isfinite(smf.pop_loss())
