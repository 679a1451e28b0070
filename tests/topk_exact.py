"""Exact-score tables for the top-k evaluators, and their float64 reference (used by test_topk_exact_cpu.py and
test_gpu_topk_exact.py).

Every score these tables produce is computed exactly by fp32, TF32 and BF16 arithmetic in any summation order, so every
kernel and path has one correct answer and the tests compare bitwise:

- 'digits' tables: item i stores the base-128 digits of a few integer sequences f_g(i) < 2^21 in groups of three
  embedding dimensions; a user row puts +-2^14, +-2^7, +-1 or 0 on the digits of one group, so its scores are +-f_g(i)
  (or a zig-zag of them).  Every product and partial sum is an integer below 2^24, and every table entry is an integer
  of at most 8 significant bits or a power of two: BF16 (round to nearest even) and TF32 packing leave them unchanged.
  Biases are integers too.
- 'bias' tables: Uw = Vw = 0 and any fp32 pattern in the item bias, which every path adds in fp32.

The reference orders each row by (score descending, id ascending) with a stable sort, excluded items at -inf (ranked
after every admissible item, lowest id first); slots beyond the catalogue get id -1 and score -inf.
"""
import numpy as np

D_MIN = 16
GROUPS = ('id', 'perm', 'plateau', 'dense')   # digit groups: dims 3g .. 3g + 2; dim 12 holds the constant 1
PLATEAU = 300
W_ASC = (2.0 ** 14, 2.0 ** 7, 1.0)

# order name -> (group, digit weights, constant term)
ORDERS = {
    'asc': ('id', W_ASC, 0.0),
    'desc': ('id', tuple(-w for w in W_ASC), 0.0),
    'zigzag': ('id', (2.0 ** 14, 2.0 ** 7, -1.0), 0.0),     # ascending blocks of 128, descending inside a block
    'const': (None, None, 0.0),
    'rand': ('perm', W_ASC, 0.0),
    'plateau': ('plateau', W_ASC, 0.0),                       # runs of 300 equal scores, ascending
    'plateau_desc': ('plateau', tuple(-w for w in W_ASC), 0.0),
    'dense': ('dense', W_ASC, 0.0),                           # 5 distinct values: tie buckets of I / 5 items
    'neg_asc': ('id', W_ASC, -2.0 ** 20),                     # every score < 0
    'neg_desc': ('id', tuple(-w for w in W_ASC), -1.0),
}


def sequences(I, seed=0):
    i = np.arange(I, dtype=np.int64)
    return {'id': i, 'perm': np.random.RandomState(seed).permutation(I).astype(np.int64), 'plateau': i // PLATEAU,
            'dense': (i // 7) % 5}


def digits_items(I, d, seed=0):
    """Vw [I, d] fp32 of a digits table (d >= D_MIN)."""
    assert d >= D_MIN and I <= 2 ** 21
    V = np.zeros((I, d), np.float32)
    for g, name in enumerate(GROUPS):
        f = sequences(I, seed)[name]
        V[:, 3 * g], V[:, 3 * g + 1], V[:, 3 * g + 2] = f >> 14, (f >> 7) & 127, f & 127
    V[:, 12] = 1.0
    return V


def digits_user(order, d):
    group, w, c = ORDERS[order]
    u = np.zeros(d, np.float32)
    if group is not None:
        g = GROUPS.index(group)
        u[3 * g:3 * g + 3] = w
    u[12] = c
    return u


def orderable_inv(o):
    """The fp32 values whose orderable key bits (hsk_topk.cuh) are `o` (uint32 array)."""
    o = np.asarray(o, np.uint32)
    u = np.where(o >> 31 == 1, o ^ np.uint32(0x80000000), o ^ np.uint32(0xFFFFFFFF)).astype(np.uint32)
    return u.view(np.float32)


def orderable(f):
    u = np.asarray(f, np.float32).view(np.uint32)
    u = np.where(u == 0x80000000, np.uint32(0), u)      # -0 == +0
    return np.where(u >> 31 == 1, u ^ np.uint32(0xFFFFFFFF), u ^ np.uint32(0x80000000)).astype(np.uint32)


def prefix_bias(I, p0=0x8080):
    """Item bias whose orderable bits are (p0 + i) << 16: one 16-bit key prefix per item (I <= 32000), ascending.  The
    default p0 starts at the smallest positive normal number, so no value depends on how a path treats denormals."""
    assert I <= 32000
    return orderable_inv((np.arange(I, dtype=np.int64) + p0).astype(np.uint32) << np.uint32(16))


def signed_zero_bias(I, seed=0):
    """+0 and -0 (a tie), with a few +-1 among them: rare enough (1 in 500) that the top 100 reach the zeros."""
    return np.random.RandomState(seed).choice(np.array([0.0, -0.0, 1.0, -1.0], np.float32), I, p=[0.499, 0.499, 0.001, 0.001])


def bf16_rne(x):
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return (r & 0xFFFFFFFF).astype(np.uint32).view(np.float32)


def tf32_rna(x):
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return (((u + 0x1000) & ~np.uint64(0x1FFF)) & 0xFFFFFFFF).astype(np.uint32).view(np.float32)


class Tables:
    """One case's fp32 tables: Uw [U, d], Vw [I, d], Ub [U] / Ib [I] / Gb [1] or None."""

    def __init__(self, Uw, Vw, Ub=None, Ib=None, Gb=None):
        self.Uw, self.Vw, self.Ub, self.Ib, self.Gb = Uw, Vw, Ub, Ib, Gb

    @property
    def d(self):
        return self.Uw.shape[1]

    def scores(self, users=None):
        """float64 scores [len(users), I] (no exclusions)."""
        U = self.Uw if users is None else self.Uw[users]
        s = U.astype(np.float64) @ self.Vw.astype(np.float64).T
        if self.Ub is not None:
            s += (self.Ub if users is None else self.Ub[users]).astype(np.float64)[:, None]
        if self.Ib is not None:
            s += self.Ib.astype(np.float64)[None, :]
        if self.Gb is not None:
            s += float(self.Gb[0])
        return s


def make_tables(kind, I, d, orders=(), biases='none', seed=0):
    """kind 'digits': one user per entry of `orders`; 'prefix' / 'zeros': bias tables with len(orders) users.
    biases: 'none', 'ib' (integer item bias) or 'all' (integer user, item and global bias); digits tables only."""
    rng = np.random.RandomState(seed + 7)
    U = len(orders)
    if kind == 'digits':
        Uw = np.stack([digits_user(o, d) for o in orders]).astype(np.float32)
        Vw = digits_items(I, d, seed)
        Ib = rng.randint(-64, 65, I).astype(np.float32) if biases in ('ib', 'all') else None
        Ub = rng.randint(-1000, 1001, U).astype(np.float32) if biases == 'all' else None
        Gb = np.array([37.0], np.float32) if biases == 'all' else None
        return Tables(Uw, Vw, Ub, Ib, Gb)
    assert biases == 'none'
    Ib = prefix_bias(I) if kind == 'prefix' else signed_zero_bias(I, seed)
    return Tables(np.zeros((U, d), np.float32), np.zeros((I, d), np.float32), None, Ib, None)


def ranked(scores):
    """Row-wise order of a float64 score matrix by (score descending, id ascending)."""
    return np.argsort(-scores, axis=1, kind='stable')


def exclusions(kind, scores, seed=0):
    """Sorted exclusion ids of one user (scores: that user's float64 row over the catalogue)."""
    I = scores.shape[0]
    rng = np.random.RandomState(seed)
    if kind == 'none':
        ex = np.zeros(0, np.int64)
    elif kind == 'rand':
        ex = rng.choice(I, min(I, max(1, I // 10)), replace=False)
    elif kind == 'top':          # exactly the highest-scoring items
        ex = ranked(scores[None, :])[0, :min(I, 500)]
    elif kind == 'edges':        # ids at tile edges
        ex = np.array([x for x in (0, 127, 128, 255, 256, I - 1) if 0 <= x < I])
    elif kind == 'allbut3':      # fewer admissible items than k: the -inf tail
        keep = rng.choice(I, min(I, 3), replace=False)
        ex = np.setdiff1d(np.arange(I), keep)
    elif kind == 'all':
        ex = np.arange(I)
    else:
        raise ValueError(kind)
    return np.unique(ex).astype(np.int32)


def csr(rows):
    indptr = np.zeros(len(rows) + 1, np.int64)
    indptr[1:] = np.cumsum([len(r) for r in rows])
    indices = np.concatenate(rows).astype(np.int32) if rows else np.zeros(0, np.int32)
    return indptr, indices


def reference_topk(scores, excl_rows, k):
    """Per user: (ids int32 [U, k], scores fp32 [U, k]) of the float64 reference.  scores: [U, I] float64; excluded
    entries are set to -inf; ties (including every -inf) resolve to the lower id; slots beyond I get -1 / -inf."""
    U, I = scores.shape
    s = scores.copy()
    for u, ex in enumerate(excl_rows):
        s[u, ex] = -np.inf
    kk = min(k, I)
    order = ranked(s)[:, :kk]
    ids = np.full((U, k), -1, np.int32)
    out = np.full((U, k), -np.inf, np.float32)
    ids[:, :kk] = order
    out[:, :kk] = np.take_along_axis(s, order, 1).astype(np.float32)
    return ids, out


def expand_rows(ref_ids, ref_scores, u_idx, n_users):
    """Reference rows of a batch: row r is user u_idx[r]'s; an invalid user index gives an empty (-1 / -inf) row."""
    Be, k = len(u_idx), ref_ids.shape[1]
    ids = np.full((Be, k), -1, np.int32)
    sc = np.full((Be, k), -np.inf, np.float32)
    ok = (u_idx >= 0) & (u_idx < n_users)
    ids[ok] = ref_ids[u_idx[ok]]
    sc[ok] = ref_scores[u_idx[ok]]
    return ids, sc
