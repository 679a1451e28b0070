"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) — numpy restatement of the ORDER CONTRACT of the deterministic
kernels (hassaku_b200/csrc/hsk_det.cu, include/hassaku_b200.h).  Every product and add is one float32 numpy operation
(rounded to nearest, never contracted into an FMA), so for the same inputs it reproduces the kernels' gradients bit for bit.

  slot s = b * N1 + j.  Item side: the B * N1 slots stably sorted by item id (equal ids keep increasing s).  User side: the
  B samples stably sorted by user id, every sample expanded to its N1 slots in j order.  A row's entries are its run of
  sorted positions P; chunks are cut at the run's ends and at every multiple of C of P.  A chunk sums from +0 in entry
  order, acc = acc + ds_s * other_row; the row is its chunk partials added in order from the first.  The global bias sums
  chunks of CG consecutive slots the same way.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np

C = 32       # kDetChunk
CG = 1024    # kDetGbChunk


def chunk_starts(keys_sorted: np.ndarray, chunk: int = C) -> np.ndarray:
    """Sorted positions where a chunk starts: a new id, or a multiple of `chunk` inside a run of one id."""
    n = len(keys_sorted)
    P = np.arange(n)
    new = np.ones(n, dtype=bool)
    new[1:] = keys_sorted[1:] != keys_sorted[:-1]
    return P[new | (P % chunk == 0)]


def segmented_rows(keys_sorted: np.ndarray, other_rows_of, ds_sorted: np.ndarray, n_rows: int, width: int,
                   chunk: int = C):
    """(rows [n_rows, width] fp32, bias [n_rows] fp32): row k = the ordered chunked sum of ds_sorted[P] * other_rows_of(P)
    over the positions P of key k.  `other_rows_of(P)` returns fp32 rows [len(P), width] (gathered on demand)."""
    n = len(keys_sorted)
    out = np.zeros((n_rows, width), dtype=np.float32)
    bias = np.zeros(n_rows, dtype=np.float32)
    if n == 0:
        return out, bias
    cs = chunk_starts(keys_sorted, chunk)
    ce = np.append(cs[1:], n)
    L = ce - cs
    acc = np.zeros((len(cs), width), dtype=np.float32)
    bacc = np.zeros(len(cs), dtype=np.float32)
    for k in range(int(L.max())):
        live = np.nonzero(L > k)[0]
        P = cs[live] + k
        d = ds_sorted[P].astype(np.float32)
        acc[live] = acc[live] + d[:, None] * other_rows_of(P)
        bacc[live] = bacc[live] + d
    # chunk partials of one key, added in order from the first
    ck = keys_sorted[cs]
    first = np.ones(len(cs), dtype=bool)
    first[1:] = ck[1:] != ck[:-1]
    head = np.nonzero(first)[0]
    n_in_key = np.diff(np.append(head, len(cs)))
    tot, btot = acc[head].copy(), bacc[head].copy()
    for r in range(1, int(n_in_key.max())):
        live = np.nonzero(n_in_key > r)[0]
        tot[live] = tot[live] + acc[head[live] + r]
        btot[live] = btot[live] + bacc[head[live] + r]
    out[ck[head]] = tot
    bias[ck[head]] = btot
    return out, bias


def ordered_chunk_sum(x: np.ndarray, chunk: int = CG) -> np.float32:
    """Sum of x (fp32) in chunks of `chunk` consecutive elements from +0, partials added in order from the first."""
    x = x.astype(np.float32).ravel()
    starts = np.arange(0, len(x), chunk)
    parts = np.zeros(len(starts), dtype=np.float32)
    for k in range(chunk):
        live = np.nonzero(starts + k < len(x))[0]
        parts[live] = parts[live] + x[starts[live] + k]
    tot = parts[0]
    for p in parts[1:]:
        tot = np.float32(tot + p)
    return tot


def scatter_grads(Uw: np.ndarray, Vw: np.ndarray, u_idx: np.ndarray, i_idx: np.ndarray, ds: np.ndarray,
                  biases=(False, False, False)) -> Dict[str, Optional[np.ndarray]]:
    """hsk_mf_scatter_grads_det on zero gradient tables: {'gU', 'gV', 'gUb', 'gIb', 'gGb'} (None where no such table).
    Uw [U, d], Vw [I, d] fp32; u_idx [B], i_idx [B, N1] int64; ds [B, N1] fp32."""
    Uw, Vw = np.asarray(Uw, np.float32), np.asarray(Vw, np.float32)
    u_idx, i_idx = np.asarray(u_idx, np.int64), np.asarray(i_idx, np.int64)
    ds = np.asarray(ds, np.float32)
    B, N1 = i_idx.shape
    d = Uw.shape[1]
    flat_i, flat_ds = i_idx.ravel(), ds.ravel()
    # item rows: slots stably sorted by item
    order = np.argsort(flat_i, kind='stable')
    gV, gIb = segmented_rows(flat_i[order], lambda P: Uw[u_idx[order[P] // N1]], flat_ds[order], Vw.shape[0], d)
    # user rows: samples stably sorted by user, expanded to their slots
    border = np.argsort(u_idx, kind='stable')
    slots = (border[:, None] * N1 + np.arange(N1)[None, :]).ravel()
    keys_u = np.repeat(u_idx[border], N1)
    gU, gUb = segmented_rows(keys_u, lambda P: Vw[flat_i[slots[P]]], flat_ds[slots], Uw.shape[0], d)
    ub, ib, gb = biases
    return {'gU': gU, 'gV': gV, 'gUb': gUb if ub else None, 'gIb': gIb if ib else None,
            'gGb': np.array([ordered_chunk_sum(flat_ds)], dtype=np.float32) if gb else None}
