"""CPU tests of packed validation's host side: argument checks of hsk_eval_topk_pack, hsk_rank_metrics_pack and
hsk_rank_metrics_sums_det_pack, the pack scratch size against the split plan, every ValueError of evaluate_mf_pack, and the
scoring-chunk rule."""
import ctypes

import pytest

SM = 148          # what the split plan assumes without a device (and a B200's SM count)
EV_CAP = 512      # candidate keys per row and split
TM, TN = 64, 128  # users / items per tile


def _plan_splits(Be, n_items, n_active):
    """eval_plan of hsk_eval.cu, restated."""
    row_tiles = (Be + TM - 1) // TM * n_active
    nt = (n_items + TN - 1) // TN
    want = SM * 2
    splits = -(-want // row_tiles) if row_tiles < want else 1
    splits = min(splits, max(nt // 16, 1), 64)
    tps = -(-nt // splits)
    return -(-nt // tps)


@pytest.mark.parametrize('Be,I,M', [(1, 1, 1), (64, 3706, 1), (64, 3706, 64), (1, 250_000, 1), (1, 250_000, 3),
                                    (1000, 250_000, 17), (8192, 250_000, 17), (64, 1_000_000, 2)])
def test_scratch_bytes_follow_the_plan(Be, I, M):
    from hassaku_b200 import _C
    got = _C.eval_topk_pack_scratch_bytes(Be, I, 100, M)
    assert got == _plan_splits(Be, I, M) * M * Be * EV_CAP * 8
    if M == 1:
        assert got == _C.eval_topk_scratch_bytes(Be, I, 100)


def test_eval_topk_pack_validates_without_gpu():
    from hassaku_b200 import _C
    lib = _C.lib()
    t = _C.MfTables(16, 4096, None, None, None, 10, 300, 4, 4)     # fake, aligned: validation fails before any launch
    ok = dict(t=ctypes.byref(t), stride=4096, n_trials=3, active=64, n_active=2, u=128, Be=8, k=100, scratch=8192,
              scratch_bytes=1 << 30)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.hsk_eval_topk_pack(a['t'], a['stride'], a['n_trials'], a['active'], a['n_active'], a['u'], a['Be'],
                                      None, None, a['k'], 256, 512, a['scratch'], a['scratch_bytes'], None, None)

    for kw, what in [(dict(t=None), b'null'), (dict(u=None), b'null'), (dict(k=0), b'k <='), (dict(k=129), b'k <='),
                     (dict(n_active=4), b'n_active'), (dict(n_active=-1), b'n_active'), (dict(n_trials=0), b'n_active'),
                     (dict(n_active=70000, n_trials=70000), b'n_active'), (dict(active=None), b'active is null'),
                     (dict(stride=6), b'trial_stride'), (dict(stride=0), b'trial_stride'),
                     (dict(scratch_bytes=100), b'scratch too small'), (dict(scratch=None), b'scratch too small'),
                     (dict(Be=1 << 30), b'n_active * Be')]:
        assert call(**kw) == -1 and what in lib.hsk_last_error(), (kw, lib.hsk_last_error())
    t_ld = _C.MfTables(16, 4096, None, None, None, 10, 300, 4, 6)
    assert call(t=ctypes.byref(t_ld)) == -1 and b'ld % 4' in lib.hsk_last_error()
    t_al = _C.MfTables(20, 4096, None, None, None, 10, 300, 4, 4)
    assert call(t=ctypes.byref(t_al)) == -1 and b'aligned' in lib.hsk_last_error()
    assert call(Be=0) == 0 and call(n_active=0) == 0      # nothing to do: no launch


def test_metrics_pack_entry_points_validate_without_gpu():
    from hassaku_b200 import _C
    lib = _C.lib()
    ks = (ctypes.c_int * 2)(10, 5)

    def metrics(top=64, k_max=10, n_trials=3, active=128, n_active=2, lab=256, ks_=ks, n_ks=2, n_groups=0):
        return lib.hsk_rank_metrics_pack(top, 8, k_max, ks_, n_ks, 512, lab, lab, None, n_groups, 1024, n_trials, active,
                                         n_active, None, 2048, 4096, None, None)

    for kw, what in [(dict(top=None), b'null'), (dict(lab=None), b'label CSR'), (dict(k_max=129), b'k_max'),
                     (dict(ks_=(ctypes.c_int * 2)(10, 11)), b'cut-off'), (dict(n_active=4), b'n_active'),
                     (dict(n_trials=0, n_active=0), b'n_active'), (dict(active=None), b'active is null'),
                     (dict(n_groups=-1), b'negative group')]:
        assert metrics(**kw) == -1 and what in lib.hsk_last_error(), (kw, lib.hsk_last_error())

    def det(per_user=64, batch=64, n_ks=4, n_trials=3, active=128, n_active=2, sums=256):
        return lib.hsk_rank_metrics_sums_det_pack(per_user, 8, batch, n_ks, 512, None, 0, n_trials, active, n_active, sums,
                                                  None, None)

    for kw, what in [(dict(per_user=None), b'null'), (dict(sums=None), b'null'), (dict(batch=0), b'batch'),
                     (dict(n_ks=9), b'n_ks'), (dict(n_active=4), b'n_active'), (dict(active=None), b'active is null')]:
        assert det(**kw) == -1 and what in lib.hsk_last_error(), (kw, lib.hsk_last_error())


# ---------------------------------------------------------------------------------------------------------------------
# evaluate_mf_pack
# ---------------------------------------------------------------------------------------------------------------------
class _Loader:
    dataset = None
    batch_size = 64


def _ev(**kw):
    from hassaku_b200.eval.eval import FullEvaluator
    return FullEvaluator(**kw)


def _raises(models, evaluators, match):
    from hassaku_b200.eval.eval import evaluate_mf_pack
    with pytest.raises(ValueError, match=match):
        evaluate_mf_pack(models, _Loader(), evaluators)


def test_evaluate_mf_pack_value_errors_name_the_condition():
    import torch
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.eval.eval import FullEvaluatorCalibrationDecorator
    a, b = SGDMatrixFactorization(30, 20, 8), SGDMatrixFactorization(30, 20, 8)
    _raises([a, b], [_ev()], 'one evaluator per model')
    _raises([a, torch.nn.Linear(2, 2)], [_ev(), _ev()], 'SGDMatrixFactorization')
    _raises([a, SGDMatrixFactorization(30, 20, 16)], [_ev(), _ev()], 'shape')
    _raises([a, SGDMatrixFactorization(30, 20, 8, use_item_bias=True)], [_ev(), _ev()], 'shape')
    b.eval_precision = 'bf16'
    _raises([a, b], [_ev(), _ev()], "eval_precision 'bf16'")
    b.eval_precision = 'fp32'
    cal = FullEvaluatorCalibrationDecorator(_ev(), torch.zeros(20, 3), torch.zeros(30, 3))
    _raises([a, b], [_ev(), cal], 'FullEvaluatorCalibrationDecorator')
    _raises([a, b], [_ev(), _ev(aggr_by_group=False)], 'aggr_by_group=False')
    _raises([a, b], [_ev(), _ev(hit=True)], 'hit=True')
    _raises([a, b], [_ev(), _ev(n_groups=2, user_to_user_group=[0] * 30)], 'n_groups')
    odd = _ev()
    odd.K_VALUES = [5, 10]
    _raises([a, b], [_ev(), odd], 'K_VALUES')
    # host models, or models with arenas of their own: not rows of one CUDA allocation
    _raises([a, b], [_ev(), _ev()], 'not a row of the')


@pytest.mark.parametrize('bs,U,I,M', [(64, 6040, 3706, 1), (64, 6040, 3706, 64), (1024, 6040, 3706, 64),
                                      (6040, 6040, 3706, 64), (64, 100, 250_000, 17), (128, 700, 300, 3), (1, 5, 10, 2)])
@pytest.mark.parametrize('budget', [1 << 20, 256 << 20])
def test_chunk_is_a_multiple_of_the_batch_within_budget(bs, U, I, M, budget):
    from hassaku_b200 import _C
    from hassaku_b200.eval.eval import pack_chunk_users
    c = pack_chunk_users(bs, U, I, 100, M, budget)
    n_batches = -(-U // bs)
    assert c % bs == 0 and bs <= c <= n_batches * bs
    size = lambda n: _C.eval_topk_pack_scratch_bytes(n, I, 100, M)
    if c > bs:
        assert size(c) <= budget
    if c < n_batches * bs:    # the largest such multiple
        assert all(size(m * bs) > budget for m in range(c // bs + 1, n_batches + 1))
