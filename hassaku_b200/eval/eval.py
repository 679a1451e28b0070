"""Full-rank evaluation behind the reference API (eval/eval.py:14-118, 211-258).

`evaluate_recommender_algorithm(alg, eval_loader, evaluator, device, verbose)` keeps its signature and returned dict,
but for an SGDMatrixFactorization the per-batch body (eval.py:243-253: [Be, I, d] broadcast product, host-side CSR
densify + H2D mask, torch.topk, 12-36 `.item()` syncs) is two kernels per user batch —
hsk_eval_topk (scoring + exclusion mask + running top-100, nothing materialised) and hsk_rank_metrics (all 12 metrics
and their per-group sums accumulated on the device) — and ONE host sync per sweep in `get_results()`.
The labels / exclusions are read straight from the dataset's CSR matrices (`iteration_matrix`, `exclude_data`,
data/dataset.py:174-191) uploaded once; the loader's dense `[Be, I]` label rows (dataset.py:199-201) are never built.
"""
import logging
from typing import Optional

import numpy as np
import torch
from tqdm import tqdm

from hassaku_b200 import _C, determinism, nvtx
from hassaku_b200.algorithms.base_classes import RecommenderAlgorithm
from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
from hassaku_b200.eval.metrics import (dense_topk, discount_table, hellinger_distance, hit_from_precision,
                                       jensen_shannon_distance, kl_divergence)

METRIC_ORDER = ('precision@{}', 'recall@{}', 'ndcg@{}')  # eval.py:78-80; column order of hsk_rank_metrics


class DeviceCSR:
    """A scipy CSR matrix as (indptr int64, indices int32) device tensors with sorted rows."""

    @classmethod
    def from_tensors(cls, indptr: torch.Tensor, indices: torch.Tensor, shape):
        """Adopt device tensors (int64 indptr [rows + 1], int32 indices sorted per row), e.g. of
        hassaku_b200.data.synthetic.make_device_interactions."""
        self = cls.__new__(cls)
        assert indptr.dtype == torch.int64 and indices.dtype == torch.int32 and indptr.numel() == shape[0] + 1
        self.shape, self.indptr, self.indices = tuple(shape), indptr.contiguous(), indices.contiguous()
        return self

    def __init__(self, m, device):
        m = getattr(m, 'm', m)  # unwrap oracle/ref_shim CsrCompat-style adapters
        m = m.tocsr()
        if not m.has_sorted_indices:
            m = m.sorted_indices()
        self.shape = m.shape
        self.indptr = torch.from_numpy(m.indptr.astype(np.int64)).to(device)
        self.indices = torch.from_numpy(m.indices.astype(np.int32)).to(device)


def device_csr(owner, attr: str, device) -> DeviceCSR:
    """Upload `getattr(owner, attr)` once per (dataset, device) and cache it on the dataset object."""
    cache = owner.__dict__.setdefault('_hsk_device_csr', {})
    key = (attr, str(device))
    if key not in cache:
        cache[key] = DeviceCSR(getattr(owner, attr), device)
    return cache[key]


class FullEvaluator:
    """Reference `FullEvaluator` (eval/eval.py:14-118): accumulates precision / recall / ndcg @ K_VALUES for the 'ALL'
    group (-1) and each user group; `get_results()` returns the means and resets.  Accumulators live on the device."""
    K_VALUES = [5, 10, 50, 100]  # eval.py:20

    def __init__(self, aggr_by_group: bool = True, n_groups: int = 0, user_to_user_group: dict = None, *,
                 hit: bool = False):
        """`hit=True` (not in the reference; keyword-only, default off so the returned dict keeps the reference's keys)
        adds `hit@k` — the share of users with at least one relevant item in the top k — next to the three metrics."""
        self.aggr_by_group = aggr_by_group
        self.n_groups = n_groups
        self.user_to_user_group = user_to_user_group
        self.hit = hit
        self._reset_internal_dict()

    def _reset_internal_dict(self):
        self._sums = None
        self._counts = None
        self._per_user = []   # (per_user [B, n_ks, 3], group [B]) when aggr_by_group is False
        self._group_dev = None
        self._hit_sums = None

    def get_n_groups(self):
        return self.n_groups

    def get_user_to_user_group(self):
        return self.user_to_user_group

    # ---- internals ----
    def _ks(self):
        return sorted(self.K_VALUES, reverse=True)

    def _prepare(self, device):
        if self._sums is None:
            n_ks = len(self.K_VALUES)
            self._sums = torch.zeros((1 + self.n_groups, n_ks, 3), dtype=torch.float64, device=device)
            self._counts = torch.zeros(1 + self.n_groups, dtype=torch.int64, device=device)
            if getattr(self, 'hit', False) and self.aggr_by_group:
                self._hit_sums = torch.zeros((1 + self.n_groups, n_ks), dtype=torch.float64, device=device)
            if self.n_groups > 0:
                g = self.user_to_user_group
                g = g if isinstance(g, torch.Tensor) else torch.as_tensor(np.asarray(g))
                self._group_dev = g.to(device=device, dtype=torch.int32).contiguous()

    def _per_user_buf(self, B, device):
        if self.aggr_by_group and not getattr(self, 'hit', False):
            return None
        return torch.empty((B, len(self.K_VALUES), 3), dtype=torch.float32, device=device)

    def _metric_outputs(self, B, device):
        """(per_user buffer or None, the sums hsk_rank_metrics adds into).  Under torch.use_deterministic_algorithms the
        kernel's atomic sums go to a discarded buffer and `_det_sums` adds the per-user rows in a fixed order."""
        per_user = self._per_user_buf(B, device)
        if not determinism.enabled():
            return per_user, self._sums
        if per_user is None:
            per_user = torch.empty((B, len(self.K_VALUES), 3), dtype=torch.float32, device=device)
        if getattr(self, '_discard', None) is None or self._discard.shape != self._sums.shape:
            self._discard = torch.zeros_like(self._sums)
        return per_user, self._discard

    def _det_sums(self, u_idxs, per_user, sums):
        if sums is not self._sums:
            _C.rank_metrics_sums_det(per_user, u_idxs, self._sums, user_group=self._group_dev, n_groups=self.n_groups)

    def _keep(self, u_idxs, per_user):
        if per_user is None:
            return
        grp = self._group_dev[u_idxs] if self.n_groups > 0 else None
        if not self.aggr_by_group:
            self._per_user.append((per_user, grp))
        elif getattr(self, 'hit', False):
            self._hit_sums = accumulate_hits(self._hit_sums, per_user, grp, self.n_groups)

    # ---- reference API: dense logits / labels (eval.py:54-99) ----
    def eval_batch(self, u_idxs: torch.Tensor, logits: torch.Tensor, y_true: torch.Tensor):
        """u_idxs [B], logits [B, n_items], y_true [B, n_items] (dense, like FullEvalDataset feeds the reference)."""
        if not logits.is_cuda:
            raise _C.HskError('FullEvaluator.eval_batch needs CUDA tensors (hassaku_b200 has no CPU path)')
        dev = logits.device
        self._prepare(dev)
        ks = self._ks()
        _, ids = dense_topk(logits, ks[0])  # eval.py:61-63
        u = u_idxs.to(dev, torch.int64).contiguous()
        y = y_true.to(dev, torch.float32).contiguous()
        per_user, sums = self._metric_outputs(len(u), dev)
        _C.rank_metrics_dense(ids, ks, u, y, discount_table(ks[0], dev), sums, self._counts,
                              user_group=self._group_dev, n_groups=self.n_groups, per_user=per_user)
        self._det_sums(u, per_user, sums)
        self._keep(u, per_user)

    # ---- fused path: ranked ids + CSR labels ----
    def eval_batch_topk(self, u_idxs: torch.Tensor, top_ids: torch.Tensor, labels: DeviceCSR):
        """u_idxs int64 [B] (device), top_ids int32 [B, 100] ranked item ids, labels = CSR of the evaluated split."""
        dev = top_ids.device
        self._prepare(dev)
        ks = self._ks()
        assert top_ids.shape[-1] == ks[0], 'Top-k indexes have different "k" compared to K_VALUES'
        per_user, sums = self._metric_outputs(len(u_idxs), dev)
        _C.rank_metrics(top_ids, ks, u_idxs, labels.indptr, labels.indices, discount_table(ks[0], dev), sums,
                        self._counts, user_group=self._group_dev, n_groups=self.n_groups, per_user=per_user)
        self._det_sums(u_idxs, per_user, sums)
        self._keep(u_idxs, per_user)

    def get_results(self):
        """eval.py:101-118 — {metric: mean over the users seen}; 'group_{g}_' prefix for user groups.  One host sync."""
        metrics_dict = dict()
        ks = self._ks()
        if self._sums is None:
            return metrics_dict
        if self.aggr_by_group:
            metrics_dict = group_means(self._sums.cpu().numpy(), self._counts.cpu().numpy(), ks, self.n_groups,
                                       self._hit_sums)
        else:
            per_user = torch.cat([p for p, _ in self._per_user]).cpu().numpy()
            grp = torch.cat([g for _, g in self._per_user]).cpu().numpy() if self.n_groups > 0 else None
            for g in range(-1, self.n_groups):
                sel = slice(None) if g == -1 else (grp == g)
                for t, k in enumerate(ks):
                    for c, name in enumerate(METRIC_ORDER):
                        key = name.format(k) if g == -1 else f'group_{g}_' + name.format(k)
                        metrics_dict[key] = per_user[sel, t, c]
                    if getattr(self, 'hit', False):
                        key = f'hit@{k}' if g == -1 else f'group_{g}_hit@{k}'
                        metrics_dict[key] = (per_user[sel, t, 0] > 0).astype(per_user.dtype)
        self._reset_internal_dict()
        return metrics_dict


def group_means(sums, counts, ks, n_groups: int, hit_sums=None) -> dict:
    """eval.py:101-118 — {metric: mean over the users seen} from one evaluator's sums [1 + n_groups, n_ks, 3] and counts
    [1 + n_groups] (host arrays; row 0 = all users, row 1 + g = user group g, 'group_{g}_' prefix)."""
    metrics_dict = dict()
    for g in range(-1, n_groups):
        for t, k in enumerate(ks):
            for c, name in enumerate(METRIC_ORDER):
                key = name.format(k) if g == -1 else f'group_{g}_' + name.format(k)
                metrics_dict[key] = float(sums[g + 1, t, c]) / int(counts[g + 1])
            if hit_sums is not None:
                key = f'hit@{k}' if g == -1 else f'group_{g}_hit@{k}'
                metrics_dict[key] = float(hit_sums[g + 1, t]) / int(counts[g + 1])
    return metrics_dict


def accumulate_hits(hit_sums: Optional[torch.Tensor], per_user: torch.Tensor, grp: Optional[torch.Tensor],
                    n_groups: int) -> torch.Tensor:
    """hit_sums [1 + n_groups, n_ks] (fp64, created on first use) += per-user hit indicators of one batch; row 0 is the
    'ALL' group, row 1 + g user group g."""
    hits = hit_from_precision(per_user).double()
    if hit_sums is None:
        hit_sums = torch.zeros((1 + n_groups, hits.shape[1]), dtype=torch.float64, device=per_user.device)
    hit_sums[0] += hits.sum(0)
    if n_groups > 0:
        hit_sums[1:].index_add_(0, grp.long(), hits)
    return hit_sums


class FullEvaluatorCalibrationDecorator(FullEvaluator):
    """Reference `FullEvaluatorCalibrationDecorator` (eval/eval.py:121-208): adds, for k in CALIBRATION_K_VALUES,
    `{prefix}_hellinger_distance@k`, `{prefix}_jensen_shannon_distance@k`, `{prefix}_kl_divergence@k` between each
    user's training distribution over tags (`user_tag_mtx[u]`) and the distribution of the top-k recommended items
    (mean of `item_tag_mtx` rows, smoothed with `beta_smoothening` of the training distribution, Steck eq. 5).
    Decorators nest (sweep_test.py:68-69: 'tag' then 'pop').  It consumes the ranked ids the wrapped evaluator already
    has: the fused path (`eval_batch_topk`) computes no second top-k; sums live on the device until `get_results()`."""
    CALIBRATION_K_VALUES = [5, 10, 50, 100]
    _NAMES = ('hellinger_distance@{}', 'jensen_shannon_distance@{}', 'kl_divergence@{}')
    _MAX_GATHER_BYTES = 256 << 20   # item_tag_mtx[top ids] is [B, k, n_tags] fp32: chunk the users above this

    def __init__(self, full_evaluator: FullEvaluator, item_tag_mtx: torch.Tensor, user_tag_mtx: torch.Tensor,
                 metric_name_prefix: str = 'tag', beta_smoothening: float = .01):
        assert 0 <= beta_smoothening <= 1, 'Beta value out of bounds'
        self.full_evaluator = full_evaluator
        self.item_tag_mtx = item_tag_mtx
        self.user_tag_mtx = user_tag_mtx
        self.metric_name_prefix = metric_name_prefix
        self.beta_smoothening = beta_smoothening
        self._cal_reset()

    @property
    def aggr_by_group(self):
        return self.full_evaluator.aggr_by_group

    @property
    def K_VALUES(self):
        return self.full_evaluator.K_VALUES

    def _cal_reset(self):
        self._cal_sums = None
        self._cal_counts = None
        self._cal_per_user = []
        self._cal_group = None

    def _reset_internal_dict(self):
        self.full_evaluator._reset_internal_dict()
        self._cal_reset()

    def get_n_groups(self):
        return self.full_evaluator.get_n_groups()

    def get_user_to_user_group(self):
        return self.full_evaluator.get_user_to_user_group()

    def _cal_ks(self):
        return sorted(self.CALIBRATION_K_VALUES, reverse=True)

    def _calibration(self, u_idxs: torch.Tensor, top_ids: torch.Tensor):
        dev = top_ids.device
        ks, G = self._cal_ks(), self.get_n_groups()
        assert top_ids.shape[-1] >= ks[0], 'Top-k indexes are shorter than the largest calibration k'
        self.user_tag_mtx = self.user_tag_mtx.to(dev)
        self.item_tag_mtx = self.item_tag_mtx.to(dev)
        if self._cal_sums is None:
            self._cal_sums = torch.zeros((1 + G, len(ks), 3), dtype=torch.float64, device=dev)
            self._cal_counts = torch.zeros(1 + G, dtype=torch.int64, device=dev)
            if G > 0:
                g = self.get_user_to_user_group()
                g = g if isinstance(g, torch.Tensor) else torch.as_tensor(np.asarray(g))
                self._cal_group = g.to(device=dev, dtype=torch.int64)
        u = u_idxs.to(dev, torch.int64)
        B, T = len(u), self.item_tag_mtx.shape[-1]
        res = torch.empty((B, len(ks), 3), dtype=torch.float32, device=dev)
        if dev.type == 'cuda':
            # one pass over each user's ranked list (hsk_topk_tag_means) instead of the [B, k, T] gather
            p = self.user_tag_mtx[u]
            tag = self.item_tag_mtx if self.item_tag_mtx.dtype == torch.float32 else self.item_tag_mtx.float()
            q_all = _C.topk_tag_means(top_ids[:, :ks[0]].to(torch.int32).contiguous(), tag.contiguous(), ks).to(p.dtype)
            for t, k in enumerate(ks):
                q = self.beta_smoothening * p + (1 - self.beta_smoothening) * q_all[:, t]      # eval.py:180-182
                res[:, t, 0] = hellinger_distance(p, q)
                res[:, t, 1] = jensen_shannon_distance(p, q)
                res[:, t, 2] = kl_divergence(p, q)                                              # target first (eval.py:192)
        chunk = max(1, min(B, self._MAX_GATHER_BYTES // max(1, ks[0] * T * 4)))
        for s in range(0, B if dev.type != 'cuda' else 0, chunk):    # host tensors (stub evaluators in the CPU tests): torch ops
            p = self.user_tag_mtx[u[s:s + chunk]]                               # training distribution [b, T]
            rows = self.item_tag_mtx[top_ids[s:s + chunk, :ks[0]].long()]        # [b, k_max, T]
            for t, k in enumerate(ks):
                q = rows[:, :k].sum(1) / k                                       # recommendation distribution
                q = self.beta_smoothening * p + (1 - self.beta_smoothening) * q  # eval.py:180-182
                res[s:s + chunk, t, 0] = hellinger_distance(p, q)
                res[s:s + chunk, t, 1] = jensen_shannon_distance(p, q)
                res[s:s + chunk, t, 2] = kl_divergence(p, q)                     # target distribution first (eval.py:192)
        grp = self._cal_group[u] if G > 0 else None
        if self.aggr_by_group:
            self._cal_sums[0] += res.double().sum(0)
            self._cal_counts[0] += B
            if G > 0:
                self._cal_sums[1:].index_add_(0, grp, res.double())
                self._cal_counts[1:] += torch.bincount(grp, minlength=G)[:G]
        else:
            self._cal_per_user.append((res, grp))

    def eval_batch(self, u_idxs: torch.Tensor, logits: torch.Tensor, y_true: torch.Tensor):
        self.full_evaluator.eval_batch(u_idxs, logits, y_true)
        if logits.is_cuda:
            _, ids = dense_topk(logits, self._cal_ks()[0])
        else:   # host tensors only reach this when the wrapped evaluator accepts them (tests with a stub evaluator)
            ids = logits.topk(self._cal_ks()[0]).indices
        self._calibration(u_idxs, ids)

    def eval_batch_topk(self, u_idxs: torch.Tensor, top_ids: torch.Tensor, labels: DeviceCSR):
        self.full_evaluator.eval_batch_topk(u_idxs, top_ids, labels)
        self._calibration(u_idxs, top_ids)

    def get_results(self):
        metrics_dict = self.full_evaluator.get_results()
        ks, G = self._cal_ks(), self.get_n_groups()
        if self._cal_sums is not None:
            if self.aggr_by_group:
                sums, counts = self._cal_sums.cpu().numpy(), self._cal_counts.cpu().numpy()
            else:
                per_user = torch.cat([r for r, _ in self._cal_per_user]).cpu().numpy()
                grp = torch.cat([g for _, g in self._cal_per_user]).cpu().numpy() if G > 0 else None
            for g in range(-1, G):
                for t, k in enumerate(ks):
                    for c, name in enumerate(self._NAMES):
                        key = self.metric_name_prefix + '_' + name.format(k)
                        key = key if g == -1 else f'group_{g}_' + key
                        if self.aggr_by_group:
                            metrics_dict[key] = float(sums[g + 1, t, c]) / int(counts[g + 1])
                        else:
                            metrics_dict[key] = per_user[slice(None) if g == -1 else (grp == g), t, c]
        self._cal_reset()
        return metrics_dict


def log_info_results(metrics_values: dict):
    """utilities/utils.py:29-40 of the reference."""
    for name in sorted(metrics_values):
        v = metrics_values[name]
        if np.ndim(v) == 0:
            logging.info('{:<30}{:.5f}'.format(name, v))


class TopKScorer:
    """hsk_eval_topk / hsk_eval_topk_tc for one model: owns the scratch, output buffers and (tensor-core modes) the
    packed operand copies for a fixed user-batch size.  precision: 'fp32' (exact, SIMT FFMA), 'tf32' or 'bf16'
    (tcgen05).  In the tensor-core modes the kernel ranks all items in low precision and returns its best
    k + RESCORE_MARGIN candidates, which hsk_rescore_topk scores again from the fp32 tables: the returned ids / scores
    are the fp32 evaluator's unless a true top-k item fell more than RESCORE_MARGIN ranks in the low-precision pass
    (`rescore=False` returns the raw low-precision ranking).  Call `refresh()` after the model's weights changed
    (re-packs the item table)."""
    RESCORE_MARGIN = 28

    def __init__(self, alg: SGDMatrixFactorization, batch_size: int, k: int, precision: str = 'fp32',
                 rescore: Optional[bool] = None):
        if precision not in _C.PRECISIONS:
            raise ValueError(f'eval precision {precision!r} not in {sorted(_C.PRECISIONS)}')
        self.alg, self.k, self.precision = alg, k, _C.PRECISIONS[precision]
        dev = alg.arena.device
        if rescore is None:
            rescore = bool(getattr(alg, 'eval_rescore', True))
        self.kc = min(128, k + self.RESCORE_MARGIN, alg.n_items) if (self.precision != 0 and rescore) else k
        self.rescore = self.kc > k
        if self.precision == 0:
            nbytes = _C.eval_topk_scratch_bytes(batch_size, alg.n_items, k)
        else:
            nbytes = _C.eval_topk_tc_scratch_bytes(batch_size, alg.n_items, k)
            kpad = _C.eval_tc_kpad(alg.embedding_dim, self.precision)
            dt = torch.float32 if self.precision == 1 else torch.bfloat16
            self.Uq = torch.empty((batch_size, kpad), dtype=dt, device=dev)
            self.Vq = torch.empty((alg.n_items, kpad), dtype=dt, device=dev)
            self.refresh()
        self.scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self.scores = torch.empty((batch_size, k), dtype=torch.float32, device=dev)
        self.ids = torch.empty((batch_size, k), dtype=torch.int32, device=dev)
        if self.rescore:
            self.cand_scores = torch.empty((batch_size, self.kc), dtype=torch.float32, device=dev)
            self.cand_ids = torch.empty((batch_size, self.kc), dtype=torch.int32, device=dev)
        self.batch_size = batch_size

    def refresh(self):
        if self.precision != 0:
            _C.pack_rows(self.alg.item_embeddings.weight.detach(), self.alg.embedding_dim, self.precision, out=self.Vq)

    def __call__(self, u_idxs: torch.Tensor, exclude: Optional[DeviceCSR]):
        B = len(u_idxs)
        assert B <= self.batch_size
        scores, ids = self.scores[:B], self.ids[:B]
        ex_p = exclude.indptr if exclude is not None else None
        ex_i = exclude.indices if exclude is not None else None
        alg = self.alg
        if self.precision == 0:
            _C.eval_topk(alg._tables(), u_idxs, self.k, scores, ids, self.scratch, ex_p, ex_i, status=alg._status())
        else:
            Uq = self.Uq[:B]
            _C.pack_rows(alg.user_embeddings.weight.detach(), alg.embedding_dim, self.precision, row_idx=u_idxs, out=Uq,
                         status=alg._status())
            cs, ci = (self.cand_scores[:B], self.cand_ids[:B]) if self.rescore else (scores, ids)
            _C.eval_topk_tc(Uq, self.Vq, self.precision, u_idxs, alg.n_users, self.kc, cs, ci, self.scratch,
                            Ub=alg.user_bias.weight.detach() if alg.use_user_bias else None,
                            Ib=alg.item_bias.weight.detach() if alg.use_item_bias else None,
                            Gb=alg.global_bias.detach() if alg.use_global_bias else None,
                            excl_indptr=ex_p, excl_indices=ex_i, status=alg._status())
            if self.rescore:
                _C.rescore_topk(alg._tables(), u_idxs, ci, self.k, scores, ids, status=alg._status(), cand_scores=cs)
        return scores, ids


_FACTOR_ATTRS = (('users_factors', 'items_factors'), ('X', 'C'))   # SVDAlgorithm / AlternatingLeastSquare; RBMF


def _cat_last(*xs):
    return torch.cat(xs, dim=-1)


# SGD models of the reference whose `combine_user_item_representations` is a dot product of per-user and per-item
# vectors (algorithms/sgd_alg.py:262-267 ACF, :353-356 UProtoMF, :450-453 IProtoMF, :535-543 UIProtoMF): the two
# representation matrices, computed once per evaluation by the model's own methods, are the factors of a frozen MF.
# UIProtoMF's sum of two dot products is one dot product of the concatenations.
_DOT_PRODUCT_REPRESENTATIONS = {
    'ACF': lambda m, u, i: (m.get_user_representations(u), m.get_item_representations(i)[0]),
    'UProtoMF': lambda m, u, i: (m.get_user_representations(u), m.get_item_representations(i)),
    'IProtoMF': lambda m, u, i: (m.get_user_representations(u), m.get_item_representations(i)),
    'UIProtoMF': lambda m, u, i: (_cat_last(*m.get_user_representations(u)),
                                  _cat_last(*reversed(m.get_item_representations(i)))),
}


def _representation_factors(alg):
    """(user matrix [U, p], item matrix [I, p]) of a dot-product SGD model, or None."""
    fn = _DOT_PRODUCT_REPRESENTATIONS.get(type(alg).__name__)
    if fn is None or not isinstance(alg, torch.nn.Module) or isinstance(alg, SGDMatrixFactorization):
        return None
    try:
        dev = next(alg.parameters()).device
    except StopIteration:
        return None
    was_training = alg.training
    alg.eval()
    with torch.no_grad():
        uf, itf = fn(alg, torch.arange(alg.n_users, device=dev), torch.arange(alg.n_items, device=dev))
    alg.train(was_training)
    return uf.detach().float(), itf.detach().float()


def factor_model_of(alg, device='cuda') -> Optional[SGDMatrixFactorization]:
    """Fitted factor models whose `predict` is the same `[B, d] x [I, d]` dot product as the MF scorer — the reference's
    SVDAlgorithm, AlternatingLeastSquare (`users_factors`, `items_factors`; algorithms/mf_algs.py:41-49, 117-125) and
    RBMF (`X`, `C`; mf_algs.py:187-194) — as a frozen SGDMatrixFactorization shell on `device`, so that they are
    evaluated by the fused top-k kernels instead of the dense `[Be, I, d]` product.  The reference's ACF / UProtoMF /
    IProtoMF / UIProtoMF torch models are handled the same way through their representation matrices (see
    `_DOT_PRODUCT_REPRESENTATIONS`; note that their regularisation side effects only happen in `forward`, which is not
    called).  Factors are cast to fp32 (the
    reference keeps what scipy / numpy produced, usually float64).  None when `alg` is not such a model.  The shell is
    cached on the algorithm object and rebuilt when the factor arrays are replaced (a new `fit`)."""
    rep = _representation_factors(alg)
    if rep is not None and 1 <= rep[0].shape[1] <= 1024:      # trainable torch model: weights change, never cached
        shell = SGDMatrixFactorization(rep[0].shape[0], rep[1].shape[0], rep[0].shape[1])
        with torch.no_grad():
            shell.user_embeddings.weight.copy_(rep[0])
            shell.item_embeddings.weight.copy_(rep[1])
        shell.to(device)
        shell.name = f'FactorModel({getattr(alg, "name", type(alg).__name__)})'
        return shell
    for ua, ia in _FACTOR_ATTRS:
        uf, itf = getattr(alg, ua, None), getattr(alg, ia, None)
        if uf is None or itf is None or isinstance(alg, SGDMatrixFactorization):
            continue
        if getattr(uf, 'ndim', 0) != 2 or getattr(itf, 'ndim', 0) != 2 or uf.shape[1] != itf.shape[1]:
            continue
        if not 1 <= uf.shape[1] <= 1024:
            continue
        cached = alg.__dict__.get('_hsk_factor_model')
        if cached is not None and cached[0] is uf and cached[1] is itf and str(cached[2].arena.device).startswith(str(device)):
            return cached[2]
        shell = SGDMatrixFactorization(uf.shape[0], itf.shape[0], uf.shape[1])
        with torch.no_grad():
            shell.user_embeddings.weight.copy_(torch.as_tensor(np.asarray(uf), dtype=torch.float32))
            shell.item_embeddings.weight.copy_(torch.as_tensor(np.asarray(itf), dtype=torch.float32))
        shell.to(device)
        shell.name = f'FactorModel({getattr(alg, "name", type(alg).__name__)})'
        alg.__dict__['_hsk_factor_model'] = (uf, itf, shell)
        return shell
    return None


def evaluate_mf_sweep(alg: SGDMatrixFactorization, labels: DeviceCSR, exclude: Optional[DeviceCSR], evaluator: FullEvaluator,
                      n_users: int, batch_size: int = 8192, verbose: bool = False, user_batches=None):
    """The SGD branch of evaluate_recommender_algorithm (eval/eval.py:237-253) on device-resident CSR matrices: per user
    batch one scoring + mask + top-k launch (TopKScorer; precision = `alg.eval_precision`, default fp32-exact) and one
    metrics launch; the accumulators stay on the device (the caller reads them with evaluator.get_results()).
    `user_batches` (optional): an iterable of int64 user-id tensors (host or device) instead of arange(n_users) in
    batches — host tensors are copied to the device per batch, like the reference loader's u_idxs."""
    dev = alg.arena.device
    if alg.n_items < max(evaluator.K_VALUES):
        raise RuntimeError('selected index k out of range')  # what torch.topk raises in the reference (eval.py:63)
    scorer = TopKScorer(alg, min(batch_size, n_users), max(evaluator.K_VALUES), getattr(alg, 'eval_precision', 'fp32'))
    if user_batches is None:
        starts = range(0, n_users, batch_size)
        user_batches = (torch.arange(s, min(s + batch_size, n_users), dtype=torch.int64, device=dev)
                        for s in (tqdm(starts) if verbose else starts))
    with torch.no_grad(), nvtx.range('hsk.eval_sweep'):
        for u_idxs in user_batches:
            with nvtx.range('hsk.eval_batch'):
                u_idxs = u_idxs.to(dev, torch.int64, non_blocking=True)
                _, ids = scorer(u_idxs, exclude)
                evaluator.eval_batch_topk(u_idxs, ids, labels)
    alg.check_status()


def evaluate_recommender_algorithm(alg: RecommenderAlgorithm, eval_loader, evaluator: FullEvaluator, device='cpu',
                                   verbose=False):
    """Evaluation procedure that calls FullEvaluator on the dataset (eval/eval.py:211-258)."""
    dataset = eval_loader.dataset
    if not isinstance(alg, SGDMatrixFactorization):
        alg = factor_model_of(alg) or alg      # SVD / ALS / RBMF: same contraction, same kernels
    if isinstance(alg, SGDMatrixFactorization):
        if not alg.arena.is_cuda:  # the reference's run_test evaluates with device='cpu' (experiment_helper.py:116)
            alg.to('cuda')
        dev = alg.arena.device
        labels = device_csr(dataset, 'iteration_matrix', dev)
        exclude = device_csr(dataset, 'exclude_data', dev)
        bs = getattr(eval_loader, 'batch_size', None) or 8192
        evaluate_mf_sweep(alg, labels, exclude, evaluator, dataset.n_users, bs, verbose=verbose)
    else:
        # generic algorithms (eval.py:224-236): `predict` runs where the algorithm lives — numpy / scipy models (KNN, SLIM,
        # EASE, pop) index host arrays with the loader's CPU tensors, torch models get tensors on their parameters'
        # device — exactly as the reference calls it; only the returned scores go to the GPU, where masking, top-k and the
        # metrics run (eval_batch)
        dev = torch.device('cuda' if str(device) == 'cpu' else device)
        alg_dev = torch.device('cpu')
        if isinstance(alg, torch.nn.Module):
            alg_dev = next((p.device for p in alg.parameters()), torch.device(device))
        exclude = getattr(dataset.exclude_data, 'm', dataset.exclude_data)
        for u_idxs, i_idxs, labels in (tqdm(eval_loader) if verbose else eval_loader):
            out = alg.predict(u_idxs.to(alg_dev), i_idxs.to(alg_dev))
            if not isinstance(out, torch.Tensor):
                out = torch.as_tensor(np.asarray(out))
            out = out.to(dev, torch.float32)
            batch_mask = torch.from_numpy(exclude[u_idxs.cpu().numpy()].toarray().astype(bool)).to(dev)
            out[batch_mask] = -torch.inf
            evaluator.eval_batch(u_idxs.to(dev), out, labels.to(dev))

    metrics_values = evaluator.get_results()
    log_info_results(metrics_values)
    return metrics_values


PACK_SCRATCH_BYTES = 256 << 20   # top-k candidate scratch of one packed scoring launch (evaluate_mf_pack)


def pack_chunk_users(batch_size: int, n_users: int, n_items: int, k: int, n_active: int,
                     budget: int = PACK_SCRATCH_BYTES) -> int:
    """Users per packed scoring launch: the largest multiple of the loader's batch size (up to the batches that cover
    n_users) whose hsk_eval_topk_pack scratch for n_active trials fits `budget`, and never less than one batch."""
    n_batches = max(1, -(-n_users // batch_size))
    per_row = _C.eval_topk_pack_scratch_bytes(1, 1, k, 1)   # one candidate list: the scratch is at least rows x this
    m = max(1, min(n_batches, budget // (per_row * n_active * batch_size)))
    while m > 1 and _C.eval_topk_pack_scratch_bytes(m * batch_size, n_items, k, n_active) > budget:
        m -= 1
    return m * batch_size


def _check_pack(models, evaluators):
    """ValueError naming the condition unless `models` are SGDMatrixFactorization of one shape with fp32 evaluation and
    `evaluators` one plain FullEvaluator per model (aggr_by_group=True, hit=False) with one K_VALUES and n_groups."""
    shape = lambda m: (m.n_users, m.n_items, m.embedding_dim, m.use_user_bias, m.use_item_bias, m.use_global_bias)
    if len(evaluators) != len(models):
        raise ValueError(f'one evaluator per model: {len(models)} models, {len(evaluators)} evaluators')
    for j, (m, ev) in enumerate(zip(models, evaluators)):
        if not isinstance(m, SGDMatrixFactorization):
            raise ValueError(f'model {j} is a {type(m).__name__}: packed evaluation takes SGDMatrixFactorization models')
        if shape(m) != shape(models[0]):
            raise ValueError(f'model {j} differs from model 0 in shape (n_users, n_items, embedding_dim, biases): '
                             f'{shape(m)} vs {shape(models[0])}')
        prec = getattr(m, 'eval_precision', 'fp32')
        if prec != 'fp32':
            raise ValueError(f"model {j} has eval_precision {prec!r}: packed evaluation runs the fp32 evaluator only")
        if type(ev) is not FullEvaluator:
            raise ValueError(f'evaluator {j} is a {type(ev).__name__}: packed evaluation takes plain FullEvaluator '
                             f'objects (no calibration decorators)')
        if not ev.aggr_by_group:
            raise ValueError(f'evaluator {j} has aggr_by_group=False: packed evaluation returns group means only')
        if getattr(ev, 'hit', False):
            raise ValueError(f'evaluator {j} has hit=True: packed evaluation has no hit@k')
        if list(ev.K_VALUES) != list(evaluators[0].K_VALUES) or ev.n_groups != evaluators[0].n_groups:
            raise ValueError(f'evaluator {j} differs from evaluator 0 in K_VALUES or n_groups')


def _pack_trials(models):
    """(flat [n_trials, stride] view of the allocation, trial index per model) for models whose arenas are rows of one
    [M, stride] CUDA allocation, as PackedMFTrainStep binds them; ValueError naming the condition otherwise."""
    stride = models[0].layout.n_total
    storage = models[0].arena.untyped_storage().data_ptr()
    idx = []
    for j, m in enumerate(models):
        a = m.arena
        if (not a.is_cuda or a.dtype != torch.float32 or a.dim() != 1 or a.numel() != stride or a.stride(0) != 1
                or a.untyped_storage().data_ptr() != storage or a.storage_offset() % stride != 0):
            raise ValueError(f'model {j} arena is not a row of the [M, {stride}] CUDA allocation of model 0: packed '
                             f'evaluation needs the models bound as PackedMFTrainStep binds them')
        idx.append(a.storage_offset() // stride)
    if len(set(idx)) != len(idx):
        raise ValueError('two models share one row of the allocation')
    flat = models[0].arena.detach().as_strided((max(idx) + 1, stride), (stride, 1), 0)
    return flat, idx


def evaluate_mf_pack(models, eval_loader, evaluators, device='cpu', verbose=False) -> list:
    """`[evaluate_recommender_algorithm(models[j], eval_loader, evaluators[j], device, verbose) for j]` in one packed
    sweep: per chunk of users one hsk_eval_topk_pack and one hsk_rank_metrics_pack launch for all the models, and one
    device-to-host copy for the whole sweep.  `models`: SGDMatrixFactorization of one shape whose arenas are rows of one
    [M, stride] allocation (PackedMFTrainStep binds them so; any subset, any order), fp32 evaluation; `evaluators`: plain
    FullEvaluator with aggr_by_group=True and hit=False, one per model, sharing K_VALUES and the user groups.  Anything
    else raises ValueError.

    A chunk is the largest multiple of the loader's batch size whose scratch fits PACK_SCRATCH_BYTES: a user's top-k
    list depends on that user's row alone, so the chunk does not change the ids.  Under torch.use_deterministic_algorithms
    the metric sums are taken per loader batch in order (hsk_rank_metrics_sums_det_pack), bitwise as the per-model path."""
    models, evaluators = list(models), list(evaluators)
    if not models:
        return []
    _check_pack(models, evaluators)
    flat, idx = _pack_trials(models)
    ev0, alg0 = evaluators[0], models[0]
    if alg0.n_items < max(ev0.K_VALUES):
        raise RuntimeError('selected index k out of range')  # as evaluate_mf_sweep
    dev = flat.device
    dataset = eval_loader.dataset
    labels = device_csr(dataset, 'iteration_matrix', dev)
    exclude = device_csr(dataset, 'exclude_data', dev)
    for ev in evaluators:
        ev._prepare(dev)
    G, ks = ev0.n_groups, ev0._ks()
    group = ev0._group_dev
    for j, ev in enumerate(evaluators[1:], 1):
        if G > 0 and not torch.equal(ev._group_dev, group):
            raise ValueError(f'evaluator {j} differs from evaluator 0 in user_to_user_group')
    M, T, n_ks, k = len(models), flat.shape[0], len(ks), ks[0]
    n_users = dataset.n_users
    bs = getattr(eval_loader, 'batch_size', None) or 8192
    chunk = pack_chunk_users(bs, n_users, alg0.n_items, k, M, PACK_SCRATCH_BYTES)
    # sums [T, 1 + G, n_ks, 3] fp64, counts [T, 1 + G] int64 and the status word in one buffer: one copy reads them all
    n_sums, n_counts = T * (1 + G) * n_ks * 3, T * (1 + G)
    acc = torch.zeros(n_sums + n_counts + 1, dtype=torch.float64, device=dev)
    sums = acc[:n_sums].view(T, 1 + G, n_ks, 3)
    counts = acc[n_sums:n_sums + n_counts].view(torch.int64).view(T, 1 + G)
    status = acc[n_sums + n_counts:].view(torch.int32)[:1]
    for j, ev in zip(idx, evaluators):        # what the evaluators already hold, as the per-model sweep would add to it
        sums[j].copy_(ev._sums)
        counts[j].copy_(ev._counts)
    det = determinism.enabled()
    metric_sums = torch.zeros_like(sums) if det else sums
    active = torch.tensor(idx, dtype=torch.int32).to(dev)
    Bc = min(chunk, n_users)
    scratch = torch.empty(_C.eval_topk_pack_scratch_bytes(Bc, alg0.n_items, k, M), dtype=torch.uint8, device=dev)
    top_s = torch.empty(M * Bc * k, dtype=torch.float32, device=dev)
    top_i = torch.empty(M * Bc * k, dtype=torch.int32, device=dev)
    per_user = torch.empty(M * Bc * n_ks * 3, dtype=torch.float32, device=dev) if det else None
    discount = discount_table(k, dev)
    tables = alg0.layout.tables(flat[0])
    starts = range(0, n_users, chunk)
    with torch.no_grad(), nvtx.range('hsk.eval_pack_sweep'):
        for s in (tqdm(starts) if verbose else starts):
            u = torch.arange(s, min(s + chunk, n_users), dtype=torch.int64, device=dev)
            Be = u.numel()
            ids = top_i[:M * Be * k].view(M, Be, k)
            _C.eval_topk_pack(tables, flat.shape[1], T, active, u, k, top_s[:M * Be * k].view(M, Be, k), ids, scratch,
                              exclude.indptr, exclude.indices, status=status)
            pu = per_user[:M * Be * n_ks * 3].view(M, Be, n_ks, 3) if det else None
            _C.rank_metrics_pack(ids, ks, u, labels.indptr, labels.indices, discount, active, metric_sums, counts,
                                 user_group=group, n_groups=G, per_user=pu, status=status)
            if det:
                _C.rank_metrics_sums_det_pack(pu, u, bs, active, sums, user_group=group, n_groups=G, status=status)
    host = acc.cpu()
    if int(host[n_sums + n_counts:].view(torch.int32)[0]) & _C.STATUS_BAD_INDEX:
        raise IndexError('index out of range in SGDMatrixFactorization (user or item index)')
    host_sums = host[:n_sums].view(T, 1 + G, n_ks, 3).numpy()
    host_counts = host[n_sums:n_sums + n_counts].view(torch.int64).view(T, 1 + G).numpy()
    out = []
    for j, ev in zip(idx, evaluators):
        ev._reset_internal_dict()
        metrics_values = group_means(host_sums[j], host_counts[j], ks, G)
        log_info_results(metrics_values)
        out.append(metrics_values)
    return out
