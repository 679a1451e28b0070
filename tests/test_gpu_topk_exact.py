"""GPU: every top-k path against the float64 reference on tables whose scores fp32, TF32 and BF16 all compute exactly
(tests/topk_exact.py), so ids AND scores must match bitwise (a score of 0 matches either sign: +0 and -0 are one score).

Paths: hsk_eval_topk (fp32); hsk_eval_topk_tc_v with the one-CTA and the CTA-pair kernel, BF16 and TF32 (d <= 256), raw
(k' = k) and re-scored through hsk_rescore_topk with k' = min(128, k + 28, I) as TopKScorer calls it; the merge paths
(item shards i mod G + hsk_topk_merge, hsk_eval_topk_tc_shards + hsk_rescore_topk_shards, hsk_rescore_scores +
hsk_topk_combine) and hsk_topk_dense.  The score orders are adversarial for the kernels' candidate lists: sorted streams
make the fill trigger fire in every tile, big tie buckets make the radix cut fall back to its exact sort, one 16-bit key
prefix per item drives the radix compaction, and users with fewer than k admissible items reach the -inf tail."""
import numpy as np
import pytest
import torch

import topk_exact as X

pytestmark = pytest.mark.gpu

PATHS = [('fp32', None, False)] + [(p, v, r) for v in ('single', 'pair') for p in ('bf16', 'tf32') for r in (False, True)]
MARGIN = 28


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t if dtype is None else t.to(dtype)).cuda()


def _table(a, ld=None):
    """fp32 [n, d] -> a [:, :d] view of [n, ld] device storage (ld % 4 == 0, as the kernels require)."""
    n, d = a.shape
    ld = ld or (d + 3) // 4 * 4
    t = torch.zeros((n, ld), dtype=torch.float32, device='cuda')
    t[:, :d] = _dev(a)
    return t[:, :d]


class Case:
    def __init__(self, tables, excl_rows):
        from hassaku_b200 import _C
        self.t, self.U, self.I = tables, tables.Uw.shape[0], tables.Vw.shape[0]
        self.Uw, self.Vw = _table(tables.Uw), _table(tables.Vw)
        self.Ub = None if tables.Ub is None else _dev(tables.Ub)
        self.Ib = None if tables.Ib is None else _dev(tables.Ib)
        self.Gb = None if tables.Gb is None else _dev(tables.Gb)
        self.set_exclusions(excl_rows)
        self.tables = _C.make_tables(self.Uw, self.Vw, self.Ub, self.Ib, self.Gb, tables.d)
        self.status = torch.zeros(1, dtype=torch.int32, device='cuda')

    def set_exclusions(self, excl_rows):
        """The exclusion CSR on the device; none at all is passed as no CSR (an empty index array has no storage)."""
        self.excl_rows, self._ref = excl_rows, {}
        indptr, indices = X.csr(excl_rows)
        self.indptr, self.indices = (_dev(indptr), _dev(indices)) if len(indices) else (None, None)

    def ref(self, k):
        if k not in self._ref:
            self._ref[k] = X.reference_topk(self.t.scores(), self.excl_rows, k)
        return self._ref[k]

    def expected(self, u_idx, k):
        return X.expand_rows(*self.ref(k), u_idx, self.U)

    def run(self, path, u_idx, k):
        from hassaku_b200 import _C
        prec, variant, rescore = path
        u = _dev(u_idx, torch.int64)
        Be = len(u_idx)
        s = torch.empty((Be, k), dtype=torch.float32, device='cuda')
        i = torch.empty((Be, k), dtype=torch.int32, device='cuda')
        if prec == 'fp32':
            scratch = torch.empty(_C.eval_topk_scratch_bytes(Be, self.I, k), dtype=torch.uint8, device='cuda')
            _C.eval_topk(self.tables, u, k, s, i, scratch, self.indptr, self.indices, status=self.status)
            return s, i
        P = _C.PRECISIONS[prec]
        kc = min(128, k + MARGIN, self.I) if rescore else k
        if rescore and kc <= k:
            return None
        Uq = _C.pack_rows(self.Uw, self.t.d, P, row_idx=u, status=self.status)
        Vq = _C.pack_rows(self.Vw, self.t.d, P)
        scratch = torch.empty(_C.eval_topk_tc_scratch_bytes(Be, self.I, kc), dtype=torch.uint8, device='cuda')
        cs = torch.empty((Be, kc), dtype=torch.float32, device='cuda')
        ci = torch.empty((Be, kc), dtype=torch.int32, device='cuda')
        _C.eval_topk_tc(Uq, Vq, P, u, self.U, kc, cs, ci, scratch, Ub=self.Ub, Ib=self.Ib, Gb=self.Gb,
                        excl_indptr=self.indptr, excl_indices=self.indices, status=self.status, variant=variant)
        if not rescore:
            return cs, ci
        _C.rescore_topk(self.tables, u, ci, k, s, i, status=self.status, cand_scores=cs)
        return s, i


def _check(got, want, what):
    s, i = got
    torch.cuda.synchronize()
    i, s = i.cpu().numpy(), s.cpu().numpy()
    wi, ws = want
    bad = np.nonzero((i != wi).any(1) | (s != ws).any(1))[0]
    assert len(bad) == 0, (f'{what}: {len(bad)} rows differ, first row {bad[0]}: ids {i[bad[0]][:12].tolist()} '
                           f'want {wi[bad[0]][:12].tolist()}; scores {s[bad[0]][:6].tolist()} want {ws[bad[0]][:6].tolist()}')


def _run_all(case, u_idx, k, paths=PATHS, bad_rows=False):
    want = case.expected(np.asarray(u_idx), k)
    for path in paths:
        if path[0] == 'tf32' and case.t.d > 256:
            continue
        case.status.zero_()
        got = case.run(path, np.asarray(u_idx), k)
        if got is None:
            continue
        _check(got, want, f'{path}')
        st = int(case.status.item())
        assert st == (1 if bad_rows else 0), (path, st)


def _batch(U, Be, layout='cycle'):
    if layout == 'cycle':
        return np.arange(Be) % U
    if layout == 'blocks':       # repeated user ids, each in a run of rows
        return (np.arange(Be) // 37) % U
    raise ValueError(layout)


# (kind, I, d, k, Be, orders, exclusions, biases, batch)
CASES = [
    # the -inf tail: fewer than k admissible items (all but 3 excluded / everything excluded)
    ('digits', 257, 16, 100, 2, ('asc', 'desc'), 'allbut3', 'none', 'cycle'),
    ('digits', 4097, 16, 128, 129, ('asc', 'rand', 'const'), 'allbut3', 'ib', 'cycle'),
    ('digits', 65537, 128, 33, 127, ('desc', 'zigzag'), 'allbut3', 'all', 'blocks'),
    ('digits', 256, 16, 7, 1, ('asc',), 'all', 'none', 'cycle'),
    ('digits', 4097, 16, 100, 255, ('rand', 'asc', 'desc'), 'all', 'all', 'cycle'),
    ('digits', 99, 16, 100, 2, ('asc', 'const'), 'allbut3', 'none', 'cycle'),          # I = k - 1
    # sorted streams: fill trigger in every tile; exclusions of exactly the top items / tile edges
    ('digits', 65537, 128, 100, 129, ('asc', 'plateau', 'zigzag'), 'top', 'none', 'cycle'),
    ('digits', 65537, 16, 128, 257, ('asc', 'desc', 'const'), 'edges', 'ib', 'cycle'),   # warp rows alternate
    ('digits', 4097, 402, 32, 255, ('asc', 'desc', 'plateau_desc', 'rand'), 'rand', 'all', 'blocks'),
    ('digits', 257, 256, 1, 127, ('desc', 'asc', 'const'), 'edges', 'none', 'cycle'),
    ('digits', 256, 16, 128, 129, ('zigzag', 'rand'), 'top', 'all', 'cycle'),
    ('digits', 255, 128, 7, 2, ('asc', 'desc'), 'rand', 'ib', 'cycle'),
    # big tie buckets (the cuts' exact-sort fallback), plateaus crossing tile and split boundaries
    ('digits', 65537, 16, 100, 1, ('dense',), 'none', 'none', 'cycle'),
    ('digits', 65537, 16, 33, 2, ('const', 'plateau'), 'rand', 'none', 'cycle'),
    ('digits', 4097, 128, 128, 257, ('dense', 'const', 'plateau'), 'edges', 'all', 'blocks'),
    # every score negative, I not a multiple of 256 (the ragged last tile's zero columns must never be candidates)
    ('digits', 4097, 16, 100, 129, ('neg_asc', 'neg_desc'), 'none', 'none', 'cycle'),
    ('digits', 257, 16, 32, 1, ('neg_desc',), 'none', 'none', 'cycle'),
    ('digits', 65537, 128, 7, 255, ('neg_asc', 'neg_desc'), 'edges', 'none', 'cycle'),
    # one 16-bit key prefix per item (radix compaction under the fill trigger)
    ('prefix', 32000, 16, 128, 129, ('-', '-'), 'none', 'none', 'cycle'),
    ('prefix', 4097, 16, 33, 2, ('-',), 'rand', 'none', 'cycle'),
    # +0 / -0 ties
    ('zeros', 4097, 16, 100, 127, ('-', '-'), 'rand', 'none', 'cycle'),
    # tiny catalogues: I = 1, I = k
    ('digits', 1, 16, 1, 2, ('asc', 'desc'), 'none', 'none', 'cycle'),
    ('digits', 1, 16, 7, 1, ('asc',), 'all', 'none', 'cycle'),
    ('digits', 32, 16, 32, 129, ('desc', 'const'), 'edges', 'all', 'cycle'),
    ('digits', 100, 16, 100, 1, ('rand',), 'none', 'ib', 'cycle'),
    ('digits', 128, 16, 128, 2, ('asc',), 'rand', 'none', 'cycle'),
]


def _case(kind, I, d, orders, excl, biases, seed=0):
    t = X.make_tables(kind, I, d, orders, biases, seed)
    s = t.scores()
    return Case(t, [X.exclusions(excl, s[u], seed + u) for u in range(len(orders))])


@pytest.mark.parametrize('kind,I,d,k,Be,orders,excl,biases,layout', CASES,
                         ids=[f'{c[0]}-I{c[1]}-d{c[2]}-k{c[3]}-B{c[4]}-{"+".join(c[5])}-{c[6]}-{c[7]}' for c in CASES])
def test_topk_paths_bitwise(kind, I, d, k, Be, orders, excl, biases, layout):
    case = _case(kind, I, d, orders, excl, biases)
    _run_all(case, _batch(len(orders), Be, layout), k)


def test_large_batch_single_split():
    """>= 148 x 128 rows: the tensor-core split plan has one split (no merge), sorted streams and the tail."""
    case = _case('digits', 4097, 128, ('asc', 'desc', 'const', 'rand', 'zigzag'), 'none', 'all')
    rows = list(case.excl_rows)
    rows[2] = X.exclusions('allbut3', case.t.scores()[2], 2)
    rows[1] = X.exclusions('top', case.t.scores()[1], 1)
    case.set_exclusions(rows)
    _run_all(case, _batch(5, 148 * 128, 'blocks'), 100)


def test_bad_user_index_rows_are_empty_and_flagged():
    case = _case('digits', 4097, 16, ('asc', 'desc', 'rand'), 'allbut3', 'all')
    u = _batch(3, 129)
    u[5], u[64], u[128] = -1, 3, -1
    _run_all(case, u, 100, bad_rows=True)


@pytest.mark.parametrize('I,k,orders', [(1_000_000, 100, ('asc', 'desc', 'rand', 'plateau')),
                                        (1_000_000, 128, ('dense', 'neg_asc', 'zigzag', 'asc'))])
def test_million_items(I, k, orders):
    case = _case('digits', I, 128, orders, 'none', 'ib')
    rows = list(case.excl_rows)
    rows[3] = X.exclusions('top', case.t.scores(np.array([3]))[0], 3)
    case.set_exclusions(rows)
    paths = [p for p in PATHS if p[0] in ('fp32', 'bf16')]
    _run_all(case, _batch(4, 257), k, paths=paths)


# ---- merge paths ----

def _shard_tables(case, G, g):
    """Items g, g + G, ... of the case as a local table (hsk_eval_topk / _tc with id_offset = g, id_stride = G)."""
    from hassaku_b200 import _C
    V = _table(case.t.Vw[g::G])
    Ib = None if case.t.Ib is None else _dev(case.t.Ib[g::G])
    return V, Ib, _C.make_tables(case.Uw, V, case.Ub, Ib, case.Gb, case.t.d)


MERGE_CASES = [
    ('digits', 4097, 16, 100, 129, ('asc', 'desc', 'const', 'rand'), 'allbut3', 'all'),
    ('digits', 65537, 128, 33, 255, ('plateau', 'zigzag', 'dense'), 'top', 'ib'),
    ('digits', 1000, 16, 128, 2, ('asc', 'desc'), 'all', 'none'),
    ('zeros', 4097, 16, 7, 127, ('-',), 'edges', 'none'),
]


@pytest.mark.parametrize('G', [3, 8])
@pytest.mark.parametrize('kind,I,d,k,Be,orders,excl,biases', MERGE_CASES)
def test_item_shards_merged(kind, I, d, k, Be, orders, excl, biases, G):
    """Item shards i mod G through hsk_eval_topk / hsk_eval_topk_tc (id_offset / id_stride), merged by hsk_topk_merge."""
    from hassaku_b200 import _C
    case = _case(kind, I, d, orders, excl, biases)
    u_idx = _batch(len(orders), Be)
    u = _dev(u_idx, torch.int64)
    want = case.expected(u_idx, k)
    for prec, variant in (('fp32', None), ('bf16', 'single'), ('tf32', 'pair')):
        parts_s = torch.empty((G, Be, k), dtype=torch.float32, device='cuda')
        parts_i = torch.empty((G, Be, k), dtype=torch.int32, device='cuda')
        for g in range(G):
            V, Ib, t = _shard_tables(case, G, g)
            n = V.shape[0]
            if prec == 'fp32':
                scratch = torch.empty(_C.eval_topk_scratch_bytes(Be, n, k), dtype=torch.uint8, device='cuda')
                _C.eval_topk(t, u, k, parts_s[g], parts_i[g], scratch, case.indptr, case.indices, id_offset=g, id_stride=G,
                             status=case.status)
            else:
                P = _C.PRECISIONS[prec]
                Uq = _C.pack_rows(case.Uw, d, P, row_idx=u)
                scratch = torch.empty(_C.eval_topk_tc_scratch_bytes(Be, n, k), dtype=torch.uint8, device='cuda')
                _C.eval_topk_tc(Uq, _C.pack_rows(V, d, P), P, u, case.U, k, parts_s[g], parts_i[g], scratch, Ub=case.Ub,
                                Ib=Ib, Gb=case.Gb, excl_indptr=case.indptr, excl_indices=case.indices, id_offset=g,
                                id_stride=G, status=case.status, variant=variant)
        s = torch.empty((Be, k), dtype=torch.float32, device='cuda')
        i = torch.empty((Be, k), dtype=torch.int32, device='cuda')
        _C.topk_merge(parts_s, parts_i, s, i)
        _check((s, i), want, f'shards {G} {prec}')
    assert int(case.status.item()) == 0


@pytest.mark.parametrize('G', [3, 8])
@pytest.mark.parametrize('kind,I,d,k,Be,orders,excl,biases', MERGE_CASES)
def test_tc_shards_and_rescore_shards(kind, I, d, k, Be, orders, excl, biases, G):
    """hsk_eval_topk_tc_shards (one launch over G item tables of unequal, ragged row counts) + hsk_rescore_topk_shards."""
    from hassaku_b200 import _C
    case = _case(kind, I, d, orders, excl, biases)
    u_idx = _batch(len(orders), Be)
    u = _dev(u_idx, torch.int64)
    want = case.expected(u_idx, k)
    tabs = [_shard_tables(case, G, g) for g in range(G)]
    rows = [V.shape[0] for V, _, _ in tabs]
    kc = min(128, k + MARGIN, I)
    for prec in ('bf16', 'tf32'):
        P = _C.PRECISIONS[prec]
        Vqs = [_C.pack_rows(V, d, P) for V, _, _ in tabs]
        Ibs = [Ib.data_ptr() if Ib is not None else 0 for _, Ib, _ in tabs]
        shards = _C.ItemShards(rows, Vq=[q.data_ptr() for q in Vqs], V=[V.data_ptr() for V, _, _ in tabs],
                               Ib=Ibs if case.Ib is not None else None)
        Uq = _C.pack_rows(case.Uw, d, P, row_idx=u)
        for kk in sorted({k, kc}):
            scratch = torch.empty(_C.eval_topk_tc_shards_scratch_bytes(Be, shards, kk), dtype=torch.uint8, device='cuda')
            cs = torch.empty((Be, kk), dtype=torch.float32, device='cuda')
            ci = torch.empty((Be, kk), dtype=torch.int32, device='cuda')
            _C.eval_topk_tc_shards(Uq, shards, P, u, case.U, kk, cs, ci, scratch, Ub=case.Ub, Gb=case.Gb,
                                   excl_indptr=case.indptr, excl_indices=case.indices, status=case.status)
            if kk == k:
                _check((cs, ci), want, f'tc_shards {G} {prec}')
            else:
                s = torch.empty((Be, k), dtype=torch.float32, device='cuda')
                i = torch.empty((Be, k), dtype=torch.int32, device='cuda')
                _C.rescore_topk_shards(case.tables, shards, u, ci, k, s, i, status=case.status, cand_scores=cs)
                _check((s, i), want, f'rescore_shards {G} {prec}')
    assert int(case.status.item()) == 0


@pytest.mark.parametrize('G', [1, 3])
@pytest.mark.parametrize('kind,I,d,k,Be,orders,excl,biases', MERGE_CASES)
def test_item_sharded_rescore_protocol(kind, I, d, k, Be, orders, excl, biases, G):
    """The item-sharded protocol at world size 1 with G shard tables on one GPU: per-shard hsk_eval_topk_tc with k' = k + 28,
    hsk_topk_merge, hsk_rescore_scores on every shard, hsk_topk_combine."""
    from hassaku_b200 import _C
    case = _case(kind, I, d, orders, excl, biases)
    u_idx = _batch(len(orders), Be)
    u = _dev(u_idx, torch.int64)
    want = case.expected(u_idx, k)
    kc = min(128, k + MARGIN, -(-I // G))
    if kc <= k:
        pytest.skip('no re-scoring margin')
    P = _C.PRECISIONS['bf16']
    Uq = _C.pack_rows(case.Uw, d, P, row_idx=u)
    tabs = [_shard_tables(case, G, g) for g in range(G)]
    cs = torch.empty((G, Be, kc), dtype=torch.float32, device='cuda')
    ci = torch.empty((G, Be, kc), dtype=torch.int32, device='cuda')
    for g, (V, Ib, _) in enumerate(tabs):
        scratch = torch.empty(_C.eval_topk_tc_scratch_bytes(Be, V.shape[0], kc), dtype=torch.uint8, device='cuda')
        _C.eval_topk_tc(Uq, _C.pack_rows(V, d, P), P, u, case.U, kc, cs[g], ci[g], scratch, Ub=case.Ub, Ib=Ib, Gb=case.Gb,
                        excl_indptr=case.indptr, excl_indices=case.indices, id_offset=g, id_stride=G, status=case.status)
    mcs = torch.empty((Be, kc), dtype=torch.float32, device='cuda')
    mci = torch.empty((Be, kc), dtype=torch.int32, device='cuda')
    _C.topk_merge(cs, ci, mcs, mci)
    sc = torch.empty((G, Be, kc), dtype=torch.float32, device='cuda')
    for g, (_, _, t) in enumerate(tabs):
        _C.rescore_scores(t, u, mci, sc[g], id_offset=g, id_stride=G, status=case.status)
    s = torch.empty((Be, k), dtype=torch.float32, device='cuda')
    i = torch.empty((Be, k), dtype=torch.int32, device='cuda')
    _C.topk_combine(sc, mci, k, s, i, cand_scores=mcs)
    _check((s, i), want, f'combine G={G}')
    assert int(case.status.item()) == 0


# ---- dense logits ----

@pytest.mark.parametrize('n_cols,k,orders,pad', [
    (1_000_000, 100, ('asc', 'desc', 'const', 'plateau', 'dense', 'neg_asc', 'zigzag', 'rand'), 3),
    (4097, 128, ('asc', 'desc', 'const', 'plateau_desc'), 0),
    (257, 33, ('asc', 'dense'), 64),
    (128, 128, ('desc', 'const'), 1),
])
def test_topk_dense_rows(n_cols, k, orders, pad):
    from hassaku_b200 import _C
    t = X.make_tables('digits', n_cols, 16, orders)
    s = t.scores()
    _check_dense(_C, s, k, pad)


@pytest.mark.parametrize('kind', ['prefix', 'zeros'])
def test_topk_dense_prefix_and_signed_zero_rows(kind):
    from hassaku_b200 import _C
    t = X.make_tables(kind, 32000, 16, ('-',) * 3)
    s = t.Ib.astype(np.float64)[None, :].repeat(3, 0)
    s[1] = s[1][::-1]
    s[2] = s[2][np.random.RandomState(0).permutation(32000)]
    _check_dense(_C, s, 100, 5)


def _check_dense(_C, s, k, pad):
    rows, n = s.shape
    buf = torch.full((rows, n + pad), float('nan'), dtype=torch.float32, device='cuda')   # row_stride > n_cols
    buf[:, :n] = _dev(s.astype(np.float32))
    out_s = torch.empty((rows, k), dtype=torch.float32, device='cuda')
    out_i = torch.empty((rows, k), dtype=torch.int32, device='cuda')
    _C.topk_dense(buf[:, :n], k, out_s, out_i)
    _check((out_s, out_i), X.reference_topk(s, [np.zeros(0, np.int32)] * rows, k), f'dense {n}')


def test_topk_merge_signed_zeros():
    """-0 and +0 from different lists are one score: the tie goes to the lower id."""
    from hassaku_b200 import _C
    sc = torch.tensor([[[-0.0, -1.0]], [[0.0, -0.0]]], device='cuda')
    ids = torch.tensor([[[5, 1]], [[7, 2]]], dtype=torch.int32, device='cuda')
    s = torch.empty((1, 2), dtype=torch.float32, device='cuda')
    i = torch.empty((1, 2), dtype=torch.int32, device='cuda')
    _C.topk_merge(sc, ids, s, i)
    assert i.cpu().tolist() == [[2, 5]] and s.cpu().tolist() == [[0.0, 0.0]]
