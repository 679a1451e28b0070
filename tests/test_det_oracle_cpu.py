"""CPU checks of the numpy restatement of the deterministic kernels' order contract (oracle/det_oracle.py): its chunking
and its sums against float64 references within fp32 rounding."""
import numpy as np

from oracle import det_oracle as D


def test_chunks_cut_at_runs_and_multiples_of_c():
    keys = np.array([0] * 5 + [1] * 70 + [2] + [3] * 3)
    cs = D.chunk_starts(keys, chunk=32)
    # run of 0: [0, 5); run of 1: [5, 75) cut at 32 and 64; run of 2: [75]; run of 3: [76, 79)
    assert cs.tolist() == [0, 5, 32, 64, 75, 76]


def test_scatter_oracle_vs_float64_with_multi_chunk_rows():
    rng = np.random.RandomState(0)
    U, I, d, B, N1 = 40, 60, 7, 300, 6
    Uw = rng.randn(U, d).astype(np.float32)
    Vw = rng.randn(I, d).astype(np.float32)
    u = rng.randint(0, U, B)
    u[:100] = 3                       # one user with 600 slots: many chunks
    i = rng.randint(0, I, (B, N1))
    i[:, 0] = np.where(rng.rand(B) < 0.5, 5, i[:, 0])   # one item with ~150 + slots
    ds = rng.randn(B, N1).astype(np.float32)
    g = D.scatter_grads(Uw, Vw, u, i, ds, (True, True, True))
    gU = np.zeros((U, d)); gV = np.zeros((I, d)); gUb = np.zeros(U); gIb = np.zeros(I)
    for b in range(B):
        for j in range(N1):
            x = float(ds[b, j])
            gU[u[b]] += x * Vw[i[b, j]].astype(np.float64)
            gV[i[b, j]] += x * Uw[u[b]].astype(np.float64)
            gUb[u[b]] += x
            gIb[i[b, j]] += x
    tol = 2e-5 * B * N1 ** 0.5
    np.testing.assert_allclose(g['gU'], gU, atol=tol)
    np.testing.assert_allclose(g['gV'], gV, atol=tol)
    np.testing.assert_allclose(g['gUb'], gUb, atol=tol)
    np.testing.assert_allclose(g['gIb'], gIb, atol=tol)
    np.testing.assert_allclose(g['gGb'][0], float(ds.astype(np.float64).sum()), atol=tol)
    untouched = np.setdiff1d(np.arange(I), i)
    assert (g['gV'][untouched] == 0).all() and (g['gIb'][untouched] == 0).all()
    assert D.scatter_grads(Uw, Vw, u, i, ds)['gGb'] is None


def test_ordered_chunk_sum_is_the_stated_order():
    rng = np.random.RandomState(1)
    x = (rng.randn(2500) * 10 ** rng.uniform(-3, 3, 2500)).astype(np.float32)
    want = np.float32(0)
    parts = []
    for c0 in range(0, len(x), 1024):
        acc = np.float32(0)
        for v in x[c0:c0 + 1024]:
            acc = np.float32(acc + v)
        parts.append(acc)
    want = parts[0]
    for p in parts[1:]:
        want = np.float32(want + p)
    assert D.ordered_chunk_sum(x) == want
