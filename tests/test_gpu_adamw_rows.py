"""hsk_adamw_dense_rows and the row-stamped hsk_adamw_pack bitwise against hsk_adamw_dense on the same gradient (itself
bitwise equal to torch.optim.AdamW / Adam, tests/test_gpu_adamw.py), on values that take the slow paths of the IEEE
division and square root, over segment layouts, in graph mode and in trial packs; and one launch per call."""
import pytest
import torch

pytestmark = pytest.mark.gpu

B1, B2, EPS = 0.9, 0.999, 1e-8


def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def _assert_same(got, want, what):
    for name, a, b in zip('pmv', got, want):
        ia, ib = _bits(a), _bits(b)
        bad = int((ia != ib).sum())
        assert bad == 0, f'{what}: {name} differs in {bad} / {ia.numel()} elements, first at {int((ia != ib).nonzero()[0])}'


def _log_uniform(n, lo, hi, gen):
    """random sign, exponent uniform in [lo, hi): every binade of the range, subnormals included for lo < -126"""
    e = torch.rand(n, generator=gen, dtype=torch.float64) * (hi - lo) + lo
    x = (2.0 ** e) * (1 + torch.rand(n, generator=gen, dtype=torch.float64))
    x = torch.where(torch.rand(n, generator=gen) < 0.5, -x, x)
    return x.to(torch.float32)


# values that take the slow paths: +-0, subnormals, huge gradients (g * g overflows), tiny m with huge v (m / dn is
# subnormal), v = 0 (dn = eps), and the borders of the fast range
SPECIAL = [0.0, -0.0, 1e-45, -1e-45, 1e-40, -3e-39, 1.1754942e-38, 1e-30, -1e-30, 2.1e-22, 1e-20, 1e-8, 1e-3, 1.0,
           1e15, -1e18, 1.8e19, -1.9e19, 3e30, 1e38]


def _state(n, gen, special_share=0.35):
    """p, m, v, g: per float4 either log-uniform over a wide range or a mix of SPECIAL values (v made non-negative)"""
    out = []
    for k, (lo, hi) in enumerate([(-40, 4), (-90, 40), (-160, 70), (-90, 40)]):
        x = _log_uniform(n, lo, hi, gen)
        pick = (torch.rand(n, generator=gen) < special_share)
        pick |= (torch.rand(n // 4 + 1, generator=gen) < special_share).repeat_interleave(4)[:n]   # whole float4s too
        sp = torch.tensor(SPECIAL)[torch.randint(0, len(SPECIAL), (n,), generator=gen)]
        x = torch.where(pick, sp, x)
        if k == 2:
            x = x.abs()
            x[torch.rand(n, generator=gen) < 0.05] = -0.0
        out.append(x)
    p, m, v, g = out
    g[torch.rand(n, generator=gen) < 0.2] = 0.0
    return p, m, v, g


def _layout(kind):
    """(n, [(offset, n_rows, ld)]) of an arena"""
    if kind == 'ld4':                     # one float4 per row (magic 0), gaps before and after, scalar tail
        return 4 * 1000 + 4 * 3001 + 4 * 77 + 3, [(4000, 3001, 4)]
    if kind == 'ld128':
        return 64 + 2000 * 128 + 37, [(64, 2000, 128)]
    if kind == 'ld404':                   # 101 float4s per row: rows straddle warps and blocks
        return 404 * 1500 + 32 + 4, [(32, 1500, 404)]
    if kind == 'four':                    # 4 segments, two of them empty, padding between segments
        return 410000, [(16, 0, 4), (32, 300, 128), (32 + 300 * 128 + 32, 0, 8), (32 + 300 * 128 + 96, 900, 404)]
    if kind == 'four_full':               # 4 non-empty segments, no gaps at all
        return 4 * 10 + 8 * 20 + 128 * 30 + 404 * 40, [(0, 10, 4), (40, 20, 8), (200, 30, 128), (4040, 40, 404)]
    if kind == 'tiny':                    # smaller than one block
        return 4 * 6 + 12 * 5 + 2, [(4, 5, 12)]
    if kind == 'none':
        return 12345, []
    raise ValueError(kind)


def _stamps_and_mask(n, segs, step, gen, dev):
    """per segment a stamp array with stale values of every other step (wrapping across 255) and a share of rows with
    the stamp of `step`; returns the segments with stamps and the element mask of untouched rows"""
    from hassaku_b200 import _C
    st = _C.row_stamp(step)
    untouched = torch.zeros(n, dtype=torch.bool)
    out = []
    for off, rows, ld in segs:
        s = torch.randint(0, 256, (max(rows, 1),), generator=gen, dtype=torch.int64)
        s[s == st] = (st % 255) + 1
        hit = torch.rand(max(rows, 1), generator=gen) < 0.3
        hit[:3] = torch.tensor([True, False, True])[:max(rows, 1)]
        s[hit] = st
        s = s.to(torch.uint8)
        if rows:
            untouched[off:off + rows * ld] = (~hit[:rows]).repeat_interleave(ld)
        out.append((off, rows, ld, s.to(dev)))
    return out, untouched


def _run_rows(state, segs, lr, wd, step, arith, adam_l2, dev='cuda'):
    from hassaku_b200 import _C
    p, m, v, g = (x.clone().to(dev) for x in state)
    _C.adamw_dense_rows(p, m, v, g, segs, lr, B1, B2, EPS, wd, step, arith=arith, adam_l2=adam_l2)
    assert int((g != 0).sum()) == 0, 'the gradient is not all zero afterwards'
    return p, m, v


def _run_dense(state, lr, wd, step, arith, adam_l2, dev='cuda'):
    from hassaku_b200 import _C
    p, m, v, g = (x.clone().to(dev) for x in state)
    _C.adamw_dense(p, m, v, g, lr, B1, B2, EPS, wd, step, arith=arith, adam_l2=adam_l2, zero_grad=True)
    return p, m, v


MODES = [('adamw', 3e-4, 4e-5), ('adamw', 1e-3, 0.0), ('adam', 1e-3, 1e-4), ('adam', 1e-3, 0.0)]


@pytest.mark.parametrize('arith', [0, 1])
@pytest.mark.parametrize('opt_name,lr,wd', MODES)
@pytest.mark.parametrize('step', [1, 4321])
def test_slow_path_values_bitwise(arith, opt_name, lr, wd, step):
    """special and wide-range values, stamped and unstamped rows mixed inside every warp's range (ld 4 and ld 12)"""
    gen = torch.Generator().manual_seed(step * 10 + arith)
    n = 4 * 50000 + 12 * 20000 + 64 + 2
    segs = [(64, 50000, 4), (64 + 4 * 50000, 20000, 12)]
    segs, untouched = _stamps_and_mask(n, segs, step, gen, 'cuda')
    state = list(_state(n, gen))
    state[3][untouched] = 0.0             # the contract: g is zero in rows not stamped this step
    got = _run_rows(state, segs, lr, wd, step, arith, opt_name == 'adam')
    want = _run_dense(state, lr, wd, step, arith, opt_name == 'adam')
    _assert_same(got, want, f'{opt_name} wd={wd} arith={arith} step={step}')


@pytest.mark.parametrize('kind', ['ld4', 'ld128', 'ld404', 'four', 'four_full', 'tiny', 'none'])
@pytest.mark.parametrize('step', [3, 254, 255, 256, 510])
def test_layouts_bitwise(kind, step):
    gen = torch.Generator().manual_seed(step + 7)
    n, segs = _layout(kind)
    segs, untouched = _stamps_and_mask(n, segs, step, gen, 'cuda')
    state = list(_state(n, gen, special_share=0.1))
    state[3][untouched] = 0.0
    for arith, (opt_name, lr, wd) in [(0, MODES[0]), (1, MODES[2])]:
        got = _run_rows(state, segs, lr, wd, step, arith, opt_name == 'adam')
        want = _run_dense(state, lr, wd, step, arith, opt_name == 'adam')
        _assert_same(got, want, f'{kind} step={step} arith={arith}')


@pytest.mark.parametrize('opt_name,lr,wd', [('adamw', 3e-4, 4e-5), ('adam', 1e-3, 1e-4)])
def test_vs_torch_adamw_foreach(opt_name, lr, wd):
    """three steps from zero state against torch.optim.AdamW / Adam (foreach) on CUDA, special p and g values"""
    from hassaku_b200 import _C
    gen = torch.Generator().manual_seed(5)
    n, segs0 = _layout('ld404')
    p0 = _state(n, gen, special_share=0.2)[0]
    p = p0.clone().cuda()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    tp = torch.nn.Parameter(p0.clone().cuda())
    opt = (torch.optim.AdamW if opt_name == 'adamw' else torch.optim.Adam)([tp], lr=lr, weight_decay=wd, foreach=True)
    for step in (1, 2, 3):
        segs, untouched = _stamps_and_mask(n, segs0, step, gen, 'cuda')
        g = _state(n, gen, special_share=0.2)[3]
        g[untouched] = 0.0
        gd = g.cuda()
        _C.adamw_dense_rows(p, m, v, gd, segs, lr, B1, B2, EPS, wd, step, arith=0, adam_l2=opt_name == 'adam')
        tp.grad = g.cuda()
        opt.step()
        st = opt.state[tp]
        _assert_same((p, m, v), (tp.detach(), st['exp_avg'], st['exp_avg_sq']), f'{opt_name} step {step}')


def _consts_dev(lr, wd, step):
    from hassaku_b200 import _C
    h = torch.empty(8, dtype=torch.float32)
    _C.adamw_consts(lr, B1, B2, EPS, wd, step, h)
    return h.cuda()


@pytest.mark.parametrize('adam_l2', [False, True])
def test_graph_mode_direct(adam_l2):
    """consts_dev / step_dev against hsk_adamw_dense_graph, and (AdamW, wd != 0) against the host-constant form"""
    from hassaku_b200 import _C
    gen = torch.Generator().manual_seed(11)
    n, segs0 = _layout('four')
    lr, wd = 1e-3, 4e-5
    for step in (1, 255, 3000):
        segs, untouched = _stamps_and_mask(n, segs0, step, gen, 'cuda')
        state = list(_state(n, gen))
        state[3][untouched] = 0.0
        p, m, v, g = (x.clone().cuda() for x in state)
        cd, sd = _consts_dev(lr, wd, step), torch.tensor([step], dtype=torch.int64, device='cuda')
        _C.adamw_dense_rows(p, m, v, g, segs, 0.0, 0.0, 0.0, 0.0, 0.0, step, arith=0, adam_l2=adam_l2, consts_dev=cd, step_dev=sd)
        assert int((g != 0).sum()) == 0
        rp, rm, rv, rg = (x.clone().cuda() for x in state)
        _C.adamw_dense_graph(rp, rm, rv, rg, cd, decoupled=not adam_l2, adam_l2=adam_l2, zero_grad=True)
        _assert_same((p, m, v), (rp, rm, rv), f'graph mode l2={adam_l2} step={step}')
        if not adam_l2:
            _assert_same((p, m, v), _run_rows(state, segs, lr, wd, step, 0, False), f'graph vs host step={step}')


def test_graph_mode_captured_replays():
    """one capture of hsk_adamw_dense_rows in graph mode, replayed over steps 250-259 (the stamp wraps at 255) with the
    scalars, step, stamps and gradient rewritten before each replay"""
    from hassaku_b200 import _C
    gen = torch.Generator().manual_seed(12)
    n, segs0 = _layout('ld404')
    lr, wd = 2e-3, 1e-2
    p0, m0, v0, _ = _state(n, gen, special_share=0.1)
    p, m, v = p0.cuda(), m0.cuda(), v0.cuda()
    g = torch.zeros_like(p)
    stamps = torch.zeros(segs0[0][1], dtype=torch.uint8, device='cuda')
    segs = [(segs0[0][0], segs0[0][1], segs0[0][2], stamps)]
    cd = torch.zeros(8, dtype=torch.float32, device='cuda')
    sd = torch.zeros(1, dtype=torch.int64, device='cuda')
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            _C.adamw_dense_rows(p, m, v, g, segs, 0.0, 0.0, 0.0, 0.0, 0.0, 1, arith=0, adam_l2=False, consts_dev=cd, step_dev=sd)
    torch.cuda.synchronize()
    p.copy_(p0); m.copy_(m0); v.copy_(v0)
    rp, rm, rv = p0.cuda(), m0.cuda(), v0.cuda()
    for step in range(250, 260):
        sg, untouched = _stamps_and_mask(n, segs0, step, gen, 'cuda')
        gs = _state(n, gen, special_share=0.1)[3]
        gs[untouched] = 0.0
        stamps.copy_(sg[0][3]); g.copy_(gs); cd.copy_(_consts_dev(lr, wd, step)); sd.fill_(step)
        graph.replay()
        rg = gs.cuda()
        _C.adamw_dense_graph(rp, rm, rv, rg, cd, decoupled=True, adam_l2=False, zero_grad=True)
        torch.cuda.synchronize()
        assert int((g != 0).sum()) == 0
        _assert_same((p, m, v), (rp, rm, rv), f'replay step {step}')


@pytest.mark.parametrize('adam_l2', [False, True])
def test_pack_rows_vs_per_trial(adam_l2):
    """hsk_adamw_pack with row segments against hsk_adamw_dense_rows per trial: one trial with wd = 0, one inactive"""
    from hassaku_b200 import _C
    gen = torch.Generator().manual_seed(13)
    segs0 = [(8, 300, 12), (8 + 300 * 12 + 16, 200, 404)]
    stride = 8 + 300 * 12 + 16 + 200 * 404 + 40
    lrs, wds = [1e-3, 3e-4, 2e-2, 5e-3], [0.0, 4e-5, 1e-2, 1e-3]
    M, active = 4, [3, 0, 2]
    for step in (1, 600):
        segs, untouched = _stamps_and_mask(stride, segs0, step, gen, 'cuda')
        st = [torch.stack(x) for x in zip(*[_state(stride, gen, special_share=0.15) for _ in range(M)])]
        st[3][:, untouched] = 0.0
        p, m, v, g = (x.clone().cuda() for x in st)
        consts = _C.adamw_consts_table(lrs, wds, B1, B2, EPS, step, 1)[0].cuda()
        _C.adamw_pack(p, m, v, g, torch.tensor(active, dtype=torch.int32, device='cuda'), consts, segs, step, adam_l2)
        for j in range(M):
            if j in active:
                assert int((g[j] != 0).sum()) == 0
                want = _run_rows([x[j] for x in st], segs, lrs[j], wds[j], step, 0, adam_l2)
                _assert_same((p[j], m[j], v[j]), want, f'trial {j} step {step}')
            else:
                _assert_same((p[j], m[j], v[j]), (st[0][j], st[1][j], st[2][j]), f'inactive trial {j}')
                assert torch.equal(_bits(g[j]), _bits(st[3][j]))


def test_one_launch_per_call():
    """a call with two segments, bias vectors before, between and after them and a scalar tail is one kernel launch"""
    from hassaku_b200 import _C
    from torch.profiler import ProfilerActivity, profile
    n = 40 + 1000 * 128 + 32 + 500 * 128 + 1000 + 500 + 3
    segs = [(40, 1000, 128, torch.ones(1000, dtype=torch.uint8, device='cuda')),
            (40 + 1000 * 128 + 32, 500, 128, torch.zeros(500, dtype=torch.uint8, device='cuda'))]
    p, m, v, g = (torch.rand(n, device='cuda') for _ in range(4))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _C.adamw_dense_rows(p, m, v, g, segs, 1e-3, B1, B2, EPS, 1e-2, 1, arith=0)
        torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert len(kernels) == 1, [e.name for e in kernels]
    assert 'adamw_rows_kernel' in kernels[0].name
