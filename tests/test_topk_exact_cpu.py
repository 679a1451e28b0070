"""CPU: the exact-score tables of test_gpu_topk_exact.py and their float64 reference."""
import numpy as np
import pytest

import topk_exact as X


@pytest.mark.parametrize('I,d', [(1, 16), (257, 16), (4097, 128), (65537, 402), (2 ** 21, 16)])
def test_digits_tables_survive_bf16_and_tf32_packing(I, d):
    t = X.make_tables('digits', I, d, tuple(X.ORDERS), 'all')
    for a in (t.Uw, t.Vw):
        assert np.array_equal(X.bf16_rne(a).view(np.uint32), a.view(np.uint32))
        assert np.array_equal(X.tf32_rna(a).view(np.uint32), a.view(np.uint32))
    for b in (t.Ub, t.Ib, t.Gb):      # fp32 on every path, but integers: every sum stays exact
        assert np.array_equal(b, np.round(b))


def test_packing_restatements_round():
    """The numpy restatements of the packing do round (so the test above is not vacuous)."""
    x = np.array([1.0 + 2 ** -9, 1.0 + 3 * 2 ** -9, 257.0, 1.0 + 2 ** -11, 1.0 + 2 ** -12], np.float32)
    assert X.bf16_rne(x).tolist() == [1.0, 1.0 + 2 ** -7, 256.0, 1.0, 1.0]
    assert X.tf32_rna(x).tolist() == [1.0 + 2 ** -9, 1.0 + 3 * 2 ** -9, 257.0, 1.0 + 2 ** -10, 1.0]


@pytest.mark.parametrize('biases', ['none', 'ib', 'all'])
def test_every_score_is_an_integer_below_2_24(biases):
    I = 2 ** 21
    t = X.make_tables('digits', I, 16, tuple(X.ORDERS), biases)
    s = t.scores()
    assert np.abs(s).max() < 2 ** 24 and np.array_equal(s, np.round(s))
    # the score is exact in fp32 for every summation order, so it equals its fp32 rounding
    assert np.array_equal(s.astype(np.float32).astype(np.float64), s)


def test_orders_have_the_stated_shape():
    I = 1000
    t = X.make_tables('digits', I, 16, tuple(X.ORDERS))
    s = dict(zip(X.ORDERS, t.scores()))
    i = np.arange(I)
    assert np.array_equal(s['asc'], i) and np.array_equal(s['desc'], -i)
    assert np.array_equal(s['zigzag'], (i // 128) * 128 + (127 - i % 128) - 127)
    assert np.all(s['const'] == 0)
    assert np.array_equal(np.sort(s['rand']), i) and not np.array_equal(s['rand'], i)
    assert np.array_equal(s['plateau'], i // 300)
    assert set(s['dense'].tolist()) == {0, 1, 2, 3, 4}
    assert s['neg_asc'].max() < 0 and s['neg_desc'].max() < 0
    assert np.all(np.diff(s['neg_asc']) > 0) and np.all(np.diff(s['neg_desc']) < 0)


def test_orderable_prefix_construction_is_strictly_increasing():
    b = X.prefix_bias(32000)
    assert np.all(np.isfinite(b))
    o = X.orderable(b)
    pre = o >> 16
    assert np.all(np.diff(pre.astype(np.int64)) == 1) and np.all(o & 0xFFFF == 0)
    assert np.all(np.diff(b.astype(np.float64)) > 0)           # the float order is the key order
    assert b.min() == np.float32(2.0 ** -126) and np.all(b < np.float32(2.0 ** 126))


def test_orderable_treats_signed_zeros_as_one_score():
    assert X.orderable(np.float32(-0.0)) == X.orderable(np.float32(0.0)) == 0x80000000
    x = np.array([-np.inf, -1.0, -1e-45, 0.0, 1e-45, 1.0, np.inf], np.float32)
    assert np.all(np.diff(X.orderable(x).astype(np.int64)) > 0)
    assert np.array_equal(X.orderable_inv(X.orderable(x)), x)


def test_reference_order_and_tail_on_hand_written_cases():
    s = np.array([[3.0, 5.0, 5.0, -1.0, 0.0, -0.0],
                  [1.0, 1.0, 1.0, 1.0, 1.0, 1.0],
                  [2.0, 9.0, 7.0, 9.0, 1.0, 0.0]])
    ex = [np.array([1], np.int32), np.array([0, 2, 3, 4, 5], np.int32), np.arange(6, dtype=np.int32)]
    ids, sc = X.reference_topk(s, ex, 8)
    # row 0: 5 (id 2), 3, then the tie +0 / -0 by id, -1, the excluded id 1 at -inf, then empty slots
    assert ids[0].tolist() == [2, 0, 4, 5, 3, 1, -1, -1]
    assert sc[0].tolist()[:6] == [5.0, 3.0, 0.0, 0.0, -1.0, -np.inf] and np.all(sc[0, 6:] == -np.inf)
    # row 1: one admissible item, then every excluded id, lowest first
    assert ids[1].tolist() == [1, 0, 2, 3, 4, 5, -1, -1] and sc[1, 0] == 1.0 and np.all(sc[1, 1:] == -np.inf)
    # row 2: all excluded: ids in order at -inf
    assert ids[2].tolist() == [0, 1, 2, 3, 4, 5, -1, -1] and np.all(sc[2] == -np.inf)
    ids3, _ = X.reference_topk(s[2:], [np.zeros(0, np.int32)], 3)
    assert ids3[0].tolist() == [1, 3, 2]                         # tie 9 / 9: lower id first


def test_exclusion_kinds():
    I = 1000
    s = X.make_tables('digits', I, 16, ('asc',)).scores()[0]
    assert np.array_equal(X.exclusions('top', s), np.arange(500, 1000))
    assert X.exclusions('edges', s).tolist() == [0, 127, 128, 255, 256, 999]
    assert len(X.exclusions('allbut3', s)) == I - 3 and len(X.exclusions('all', s)) == I
    r = X.exclusions('rand', s)
    assert len(r) == 100 and np.all(np.diff(r) > 0)
    indptr, indices = X.csr([np.array([3, 5], np.int32), np.zeros(0, np.int32), np.array([1], np.int32)])
    assert indptr.tolist() == [0, 2, 2, 3] and indices.tolist() == [3, 5, 1]


def test_expand_rows_gives_bad_indices_an_empty_row():
    ids = np.array([[1, 2], [3, 4]], np.int32)
    sc = np.array([[1.0, 0.0], [2.0, 1.0]], np.float32)
    e_ids, e_sc = X.expand_rows(ids, sc, np.array([1, -1, 0, 2, 1]), 2)
    assert e_ids.tolist() == [[3, 4], [-1, -1], [1, 2], [-1, -1], [3, 4]]
    assert np.all(e_sc[[1, 3]] == -np.inf)
