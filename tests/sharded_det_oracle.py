"""TEST INFRASTRUCTURE ONLY — numpy restatement of the ORDER CONTRACT of the sharded 'ordered' step
(include/hassaku_b200.h: hsk_shard_unpack_ordered, hsk_mf_train_fused_det_n), built on oracle/det_oracle.py's single-GPU
restatement.  Every add is one float32 numpy operation, so for the same inputs it reproduces the kernels' bits.

  Every rank applies the single-GPU contract to the samples whose user it owns, items keyed owner-major
  ((i % G) * cap + i // G, the compact table's order); an item row is the contributions of the ranks that fetched it
  added in increasing rank order (the first stored); the global bias is the ranks' values added in rank order from rank
  0's.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np

from hsk_testutil import ROOT  # noqa: F401  (puts the repository root on sys.path)
from oracle.det_oracle import ordered_chunk_sum, scatter_grads


def sharded_scatter_grads(Uw: np.ndarray, Vw: np.ndarray, u_idx: np.ndarray, i_idx: np.ndarray, ds_per_rank,
                          G: int, biases=(False, False, False)) -> Dict[str, Optional[np.ndarray]]:
    """The sharded 'ordered' step's gradients at the owners (order contract points 1 to 3) on zero gradient tables, as
    full tables in global ids: {'gU', 'gV', 'gUb', 'gIb', 'gGb'}.  Uw [U, d], Vw [I, d] fp32: the parameters the step
    started from; u_idx [B], i_idx [B, N1] int64: the GLOBAL batch; ds_per_rank[r] [B_r, N1] fp32: dL/ds of the samples
    rank r processes (u % G == r, in global batch order)."""
    Uw, Vw = np.asarray(Uw, np.float32), np.asarray(Vw, np.float32)
    u_idx, i_idx = np.asarray(u_idx, np.int64), np.asarray(i_idx, np.int64)
    n_items = Vw.shape[0]
    cap = -(-n_items // G)
    ids = np.arange(n_items)
    key = (ids % G) * cap + ids // G             # owner-major: the compact table's row order
    Vk = np.zeros((G * cap, Vw.shape[1]), dtype=np.float32)
    Vk[key] = Vw
    ub, ib, gb = biases
    out = {'gU': np.zeros_like(Uw), 'gV': np.zeros_like(Vw), 'gUb': np.zeros(Uw.shape[0], np.float32) if ub else None,
           'gIb': np.zeros(n_items, np.float32) if ib else None, 'gGb': None}
    fetched = np.zeros(n_items, dtype=bool)
    gb_total = None
    for r in range(G):
        sel = u_idx % G == r
        u_r, i_r = u_idx[sel], i_idx[sel]
        ds_r = np.asarray(ds_per_rank[r], np.float32).reshape(i_r.shape)
        # 1. the single-GPU contract on the rank's batch (users keyed by global id: same order as by local row)
        g = scatter_grads(Uw, Vk, u_r, key[i_r], ds_r, (ub, ib, False))
        mine = np.unique(u_r)
        out['gU'][mine] = g['gU'][mine]
        if ub:
            out['gUb'][mine] = g['gUb'][mine]
        # 2. item rows at the owners: the fetching ranks' contributions in rank order, the first stored
        rows = np.unique(i_r)
        first, later = rows[~fetched[rows]], rows[fetched[rows]]
        out['gV'][first] = g['gV'][key[first]]
        out['gV'][later] = out['gV'][later] + g['gV'][key[later]]
        if ib:
            out['gIb'][first] = g['gIb'][key[first]]
            out['gIb'][later] = out['gIb'][later] + g['gIb'][key[later]]
        fetched[rows] = True
        # 3. the global bias: rank values in rank order from rank 0's (a rank without samples contributes +0)
        v = ordered_chunk_sum(ds_r) if ds_r.size else np.float32(0.0)
        gb_total = v if gb_total is None else np.float32(gb_total + v)
    if gb:
        out['gGb'] = np.array([gb_total], dtype=np.float32)
    return out
