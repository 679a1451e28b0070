"""hsk_adamw_dense_rows_lag / hsk_adamw_lag_sync bitwise against hsk_adamw_dense_rows over multi-step runs (p after every
step, m and v after a sync; with lag 1 m and v after every step too), and DenseAdam(state_lag=K) against
DenseAdam(state_lag=1) through FusedMFTrainStep under the deterministic switch."""
import pytest
import torch

from test_gpu_adamw_rows import B1, B2, EPS, _bits, _layout, _stamps_and_mask, _state

pytestmark = pytest.mark.gpu


def _same(a, b, what):
    ia, ib = _bits(a), _bits(b)
    bad = int((ia != ib).sum())
    assert bad == 0, f'{what}: differs in {bad} / {ia.numel()} elements, first at {int((ia != ib).nonzero()[0])}'


def _bases(segs, step0):
    """per segment (base_in, base_out), every row's m / v those of step0 - 1"""
    return [[torch.full((max(rows, 1),), (step0 - 1) & 255, dtype=torch.uint8, device='cuda') for _ in range(2)]
            for _off, rows, _ld in segs]


def _run(kind, K, arith, opt_name, lr, wd, step0, n_steps, gen, special_share=0.1, sync_at=(), cold_rows=0):
    """n_steps steps from step0 on one layout: the lagged pass against hsk_adamw_dense_rows on the same gradients.
    cold_rows: the first rows of every segment never get a gradient."""
    from hassaku_b200 import _C
    n, segs0 = _layout(kind)
    p0, m0, v0, _ = _state(n, gen, special_share)
    ref = [x.cuda() for x in (p0, m0, v0)]
    got = [x.cuda() for x in (p0, m0, v0)]
    bases = _bases(segs0, step0)
    adam_l2 = opt_name == 'adam'
    for step in range(step0, step0 + n_steps):
        segs, untouched = _stamps_and_mask(n, segs0, step, gen, 'cuda')
        if cold_rows:
            segs = [(off, rows, ld, st.clone()) for off, rows, ld, st in segs]
            for (off, rows, ld, st) in segs:
                if rows:
                    st[:cold_rows] = (_C.row_stamp(step) % 255) + 1
                    untouched[off:off + min(cold_rows, rows) * ld] = True
        g = _state(n, gen, special_share)[3]
        g[untouched] = 0.0
        gr, gg = g.cuda(), g.cuda()
        _C.adamw_dense_rows(ref[0], ref[1], ref[2], gr, segs, lr, B1, B2, EPS, wd, step, arith=arith, adam_l2=adam_l2)
        _C.adamw_dense_rows_lag(got[0], got[1], got[2], gg, segs, bases, K, lr, B1, B2, EPS, wd, step, arith=arith,
                                adam_l2=adam_l2)
        for b in bases:
            b[0], b[1] = b[1], b[0]
        assert int((gg != 0).sum()) == 0, 'the gradient is not all zero afterwards'
        what = f'{kind} K={K} arith={arith} {opt_name} wd={wd} step={step}'
        _same(got[0], ref[0], what + ' p')
        if K == 1:
            _same(got[1], ref[1], what + ' m')
            _same(got[2], ref[2], what + ' v')
        if step in sync_at or step == step0 + n_steps - 1:
            _C.adamw_lag_sync(got[1], got[2], segs, bases, B1, B2, step, arith=arith)
            for b in bases:
                b[0], b[1] = b[1], b[0]
            _same(got[1], ref[1], what + ' m after sync')
            _same(got[2], ref[2], what + ' v after sync')
            for (_off, rows, _ld), b in zip(segs0, bases):
                assert rows == 0 or int((b[0][:rows] != (step & 255)).sum()) == 0, 'sync leaves every base at step'


MODES = [('adamw', 3e-4, 4e-5), ('adamw', 1e-3, 0.0), ('adam', 1e-3, 0.0)]


@pytest.mark.parametrize('K', [1, 2, 5, 8, 128])
@pytest.mark.parametrize('arith', [0, 1])
@pytest.mark.parametrize('opt_name,lr,wd', MODES)
def test_slow_path_values_multistep(K, arith, opt_name, lr, wd):
    """special values (+-0, subnormals, v = 0, g * g overflowing) over 12 steps across the stamp wrap (255) and the base
    wrap (256), with a sync in the middle"""
    gen = torch.Generator().manual_seed(K * 100 + arith * 10 + len(opt_name) + int(wd > 0))
    _run('ld128', K, arith, opt_name, lr, wd, 248, 12, gen, special_share=0.35, sync_at=(253,))


@pytest.mark.parametrize('kind', ['ld4', 'ld128', 'ld404', 'four', 'four_full', 'tiny', 'none'])
@pytest.mark.parametrize('K', [1, 5, 8])
def test_layouts_multistep(kind, K):
    gen = torch.Generator().manual_seed(K + 31)
    for arith, (opt_name, lr, wd) in [(0, MODES[0]), (1, MODES[2])]:
        _run(kind, K, arith, opt_name, lr, wd, 3, 10, gen)


@pytest.mark.parametrize('K', [5, 128])
def test_rows_untouched_for_300_steps(K):
    """the first rows of every segment never see a gradient over 320 steps (stamps and bases wrap more than once)"""
    gen = torch.Generator().manual_seed(K)
    _run('four', K, 0, 'adamw', 3e-4, 4e-5, 1, 320, gen, special_share=0.02, cold_rows=40)


def test_argument_checks():
    from hassaku_b200 import _C
    n, segs0 = _layout('ld128')
    p, m, v, g = (torch.zeros(n, device='cuda') for _ in range(4))
    segs, _ = _stamps_and_mask(n, segs0, 1, torch.Generator().manual_seed(0), 'cuda')
    bases = _bases(segs0, 1)
    with pytest.raises(_C.HskError, match='L2'):
        _C.adamw_dense_rows_lag(p, m, v, g, segs, bases, 4, 1e-3, B1, B2, EPS, 1e-4, 1, adam_l2=True)
    for K in (0, 129):
        with pytest.raises(_C.HskError, match='lag must be'):
            _C.adamw_dense_rows_lag(p, m, v, g, segs, bases, K, 1e-3, B1, B2, EPS, 1e-4, 1)
    with pytest.raises(_C.HskError, match='distinct'):
        _C.adamw_dense_rows_lag(p, m, v, g, segs, [[bases[0][0], bases[0][0]]], 4, 1e-3, B1, B2, EPS, 1e-4, 1)
    with pytest.raises(_C.HskError, match='one \\(base_in, base_out\\) pair per segment'):
        _C.adamw_dense_rows_lag(p, m, v, g, segs, [], 4, 1e-3, B1, B2, EPS, 1e-4, 1)
    # the C entry points themselves, without base arrays
    arr = _C._row_segments(segs, 'test')[1]
    for fn, args in ((_C.lib().hsk_adamw_dense_rows_lag,
                      (p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), n, arr, 1, None, None, 4, 1e-3, B1, B2, EPS,
                       1e-4, 1, 0, 0, None)),
                     (_C.lib().hsk_adamw_lag_sync,
                      (m.data_ptr(), v.data_ptr(), n, arr, 1, None, None, B1, B2, 1, 0, None))):
        assert fn(*args) != 0
        assert b'base_in and base_out are required' in _C.lib().hsk_last_error()
    with pytest.raises(ValueError):
        from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
        from hassaku_b200.train.optim import DenseAdam
        DenseAdam(SGDMatrixFactorization.on_device(100, 50, 8, use_item_bias=True), state_lag=0)


# ---- DenseAdam(state_lag=K) through FusedMFTrainStep, against state_lag=1 -------------------------------------------
SHAPE = (200_000, 100_000, 128, 1024, 50)


def _batches(n, seed):
    U, I, _d, B, N = SHAPE
    gen = torch.Generator(device='cuda').manual_seed(seed)
    out = []
    for _ in range(n):
        u = torch.randint(0, U, (B,), generator=gen, device='cuda')
        # skewed item draws: popular items are touched in most steps, the tail rarely
        i = (torch.rand((B, N + 1), generator=gen, device='cuda') ** 3 * I).long().clamp_(max=I - 1)
        out.append((u, i))
    return out


def _trainer(lag, wd=1e-2, decoupled=True, arith=0):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    U, I, d, _B, _N = SHAPE
    model = SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=5)
    opt = DenseAdam(model, lr=1e-3, weight_decay=wd, decoupled=decoupled, arith=arith, state_lag=lag)
    return model, opt, FusedMFTrainStep(model, RecBayesianPersonalizedRankingLoss(), opt)


@pytest.fixture
def det_mode():
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def _pair(lag, **kw):
    a, b = _trainer(1, **kw), _trainer(lag, **kw)
    _same(a[0].arena, b[0].arena, 'initial arena')
    return a, b


def _step_both(a, b, u, i, what):
    a[2](u, i)
    b[2](u, i)
    assert a[2].pop_loss_sum() == b[2].pop_loss_sum(), what + ' loss'
    _same(b[0].arena, a[0].arena, what + ' p')


@pytest.mark.parametrize('lag,arith', [(8, 0), (5, 1), (16, 0)])
def test_dense_adam_lag_bitwise(det_mode, lag, arith):
    batches = _batches(40, seed=lag)
    a, b = _pair(lag, arith=arith)
    for s, (u, i) in enumerate(batches):
        _step_both(a, b, u, i, f'step {s + 1}')
        assert b[1]._segments == () and len(b[1]._behind) == 2, 'the lagged path ran'
    _same(b[1].m, a[1].m, 'm')
    _same(b[1].v, a[1].v, 'v')
    assert not b[1]._behind


def test_dense_adam_lag_default_and_adam_wd0(det_mode):
    from hassaku_b200.train.optim import DEFAULT_STATE_LAG
    batches = _batches(12, seed=2)
    assert _trainer(DEFAULT_STATE_LAG)[1].state_lag == DEFAULT_STATE_LAG > 1
    a, b = _pair(DEFAULT_STATE_LAG, wd=0.0, decoupled=False)
    for s, (u, i) in enumerate(batches):
        _step_both(a, b, u, i, f'adam wd=0 step {s + 1}')
    assert b[1]._behind, 'Adam without weight decay lags'
    _same(b[1].m, a[1].m, 'm')
    _same(b[1].v, a[1].v, 'v')


def test_writes_through_m_v_views_are_honoured(det_mode):
    batches = _batches(14, seed=3)
    a, b = _pair(8)
    for s, (u, i) in enumerate(batches):
        if s in (5, 9):
            for opt in (a[1], b[1]):
                mU, mV = opt.model.layout.views(opt.m)[:2]
                vU = opt.model.layout.views(opt.v)[0]
                mU[:1000].mul_(0.5)
                mV[::7].zero_()
                vU[500:9000].add_(1e-6)
        _step_both(a, b, u, i, f'step {s + 1}')
    _same(b[1].m, a[1].m, 'm')
    _same(b[1].v, a[1].v, 'v')


def test_autograd_step_and_t_assignment_after_fused_steps(det_mode):
    """an autograd step() (dense gradients: the plain kernel) and an assignment of t after lagged steps"""
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    batches = _batches(10, seed=4)
    a, b = _pair(8)
    loss_fn = RecBayesianPersonalizedRankingLoss()
    for s, (u, i) in enumerate(batches):
        if s in (4, 7):
            for model, opt, _ in (a, b):
                model.zero_grad()
                out = model(u[:64], i[:64])
                labels = torch.zeros(out.shape, dtype=out.dtype, device='cuda')
                labels[:, 0] = 1.
                loss_fn.compute_loss(out, labels).backward()
                opt.step()
            _same(b[0].arena, a[0].arena, f'autograd step at {s}')
        if s == 8:
            a[1].t, b[1].t = 300, 300
        _step_both(a, b, u, i, f'step {s + 1}')
    _same(b[1].m, a[1].m, 'm')
    _same(b[1].v, a[1].v, 'v')


def test_betas_change_mid_run(det_mode):
    batches = _batches(12, seed=6)
    a, b = _pair(8)
    for s, (u, i) in enumerate(batches):
        if s == 6:
            for opt in (a[1], b[1]):
                opt.param_groups[0]['betas'] = (0.8, 0.99)
        _step_both(a, b, u, i, f'step {s + 1}')
    _same(b[1].m, a[1].m, 'm')
    _same(b[1].v, a[1].v, 'v')
