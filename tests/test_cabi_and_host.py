"""CPU tests: the C-ABI library loads and exports every symbol include/hassaku_b200.h declares (no compute calls
without a GPU), and the host-side logic (arena layout, API surface, datasets, batch generator, byte accounting)."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from hsk_testutil import ROOT


def _declared_symbols():
    src = open(os.path.join(ROOT, 'include', 'hassaku_b200.h')).read()
    return sorted(set(re.findall(r'HSK_API\s+[\w\s\*]+?\b(hsk_\w+)\s*\(', src)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as g
    from hassaku_b200 import _C
    if not os.path.exists(_C.LIB_PATH):
        g.build()
    declared = _declared_symbols()
    assert len(declared) >= 14
    lib = ctypes.CDLL(_C.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/hassaku_b200.h but not exported'
    assert sorted(_C.exported_symbols()) == declared, 'ctypes binding and header disagree'
    nm = subprocess.run(['nm', '-D', '--defined-only', _C.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r'\bT (hsk_\w+)', nm)))
    assert exported == declared, 'exported symbol set differs from the header'
    assert _C.lib().hsk_version() >= 100
    # no torch types / C++ mangled names cross the boundary
    assert not re.findall(r' T _Z', nm)


def test_argument_validation_without_gpu():
    from hassaku_b200 import _C
    lib = _C.lib()
    rc = lib.hsk_adamw_dense(None, None, None, None, 16, 1e-3, .9, .999, 1e-8, 0., 1, 0, 0, 1, None)
    assert rc == -1 and b'null' in lib.hsk_last_error()
    rc = lib.hsk_rec_loss(None, None, 4, 4, 0, 0., 1., None, None, None, None)
    assert rc == -1
    assert lib.hsk_eval_topk_scratch_bytes(8192, 3706, 100) >= 8192 * 256 * 8


def test_cuda_free_calls_fail_loudly():
    from hassaku_b200 import _C
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.eval.metrics import recall_at_k_batch
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    m = SGDMatrixFactorization(10, 120, 8)
    with pytest.raises(_C.HskError):
        m(torch.tensor([0]), torch.tensor([[1, 2]]))
    with pytest.raises(_C.HskError):
        RecBayesianPersonalizedRankingLoss().compute_loss(torch.zeros(2, 3), torch.zeros(2, 3, dtype=torch.float64))
    with pytest.raises(_C.HskError):
        recall_at_k_batch(torch.zeros(2, 20), torch.zeros(2, 20))


def test_trainer_rejects_cpu_device_and_unknown_optimizer():
    from hassaku_b200 import _C
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer import Trainer
    conf = {'device': 'cpu', 'lr': 1e-3, 'wd': 0., 'optimizer': 'adamw', 'n_epochs': 2, 'optimizing_metric': 'ndcg@10',
            'max_patience': 1, 'model_path': '/tmp', 'running_settings': {'use_wandb': False, 'batch_verbose': False}}
    with pytest.raises(_C.HskError):
        Trainer(SGDMatrixFactorization(10, 120, 8), [], [], RecBayesianPersonalizedRankingLoss(), conf)


@pytest.mark.parametrize('d', [402, 128, 7, 100])
def test_arena_layout_and_parameter_views(d):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization, ArenaLayout
    U, I = 37, 123
    lay = ArenaLayout(U, I, d, True, True, True)
    assert lay.ld % 4 == 0 and lay.ld >= d and lay.ld - d < 4
    for off in (lay.off_U, lay.off_V, lay.off_Ub, lay.off_Ib, lay.off_Gb):
        assert off % 32 == 0  # 128-byte aligned segments
    torch.manual_seed(0)
    m = SGDMatrixFactorization(U, I, d, True, True, True)
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {
        'global_bias': (1,), 'user_embeddings.weight': (U, d), 'item_embeddings.weight': (I, d),
        'user_bias.weight': (U, 1), 'item_bias.weight': (I, 1)}
    # parameters alias the arena; pad columns are zero
    Uw = m.arena[lay.off_U:lay.off_U + U * lay.ld].view(U, lay.ld)
    assert torch.equal(Uw[:, :d], m.user_embeddings.weight.detach())
    assert float(Uw[:, d:].abs().sum()) == 0.0
    with torch.no_grad():
        m.user_embeddings.weight[3, 2] = 7.
    assert float(Uw[3, 2]) == 7.


def test_same_seed_gives_reference_identical_init_and_state_dict_interop():
    """Same module construction / init order as the reference (sgd_alg.py:127-138, train/utils.py:11-13): the oracle
    model (bit-exact vs the reference, tests/test_oracle_golden.py) built from the same seed has identical weights."""
    from oracle.mf_oracle import OracleMF
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    torch.manual_seed(64)
    a = SGDMatrixFactorization(50, 130, 18, True, True, True)
    torch.manual_seed(64)
    b = OracleMF(50, 130, 18, True, True, True)
    sa, sb = a.state_dict(), b.state_dict()
    assert sorted(sa) == sorted(sb)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    # std of the init: embeddings 0.1 / d, biases 0.1 (train/utils.py:13)
    assert abs(float(sa['item_bias.weight'].std()) - 0.1) < 0.03
    b2 = OracleMF(50, 130, 18, True, True, True)
    b2.load_state_dict(sa)  # our checkpoint loads into the reference-shaped model ...
    a2 = SGDMatrixFactorization(50, 130, 18, True, True, True)
    a2.load_state_dict(b2.state_dict())  # ... and back
    for k in sa:
        assert torch.equal(a2.state_dict()[k], sa[k])
    with tempfile.TemporaryDirectory() as tmp:
        a.save_model_to_path(tmp)
        a2.load_model_from_path(tmp)
        assert os.path.exists(os.path.join(tmp, 'model.pth'))


def test_api_surface_matches_reference_names():
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.eval.eval import FullEvaluator, evaluate_recommender_algorithm  # noqa: F401
    from hassaku_b200.eval import metrics
    from hassaku_b200.train.rec_losses import RecommenderSystemLossesEnum
    from hassaku_b200.train.trainer import Trainer
    assert [e.name for e in RecommenderSystemLossesEnum] == ['bce', 'bpr', 'sampled_softmax']
    assert FullEvaluator.K_VALUES == [5, 10, 50, 100]
    for fn in ('recall_at_k_batch', 'precision_at_k_batch', 'ndcg_at_k_batch'):
        assert callable(getattr(metrics, fn))
    for meth in ('forward', 'get_user_representations', 'get_item_representations',
                 'combine_user_item_representations', 'predict', 'get_and_reset_other_loss', 'save_model_to_path',
                 'load_model_from_path', 'build_from_conf'):
        assert hasattr(SGDMatrixFactorization, meth)
    assert hasattr(Trainer, 'fit') and hasattr(Trainer, 'val')
    m = SGDMatrixFactorization(10, 120, 8)
    assert m.name == 'SGDMatrixFactorization'
    assert float(m.get_and_reset_other_loss()['reg_loss']) == 0.0

    class DS:
        n_users, n_items = 10, 120

    m2 = SGDMatrixFactorization.build_from_conf(
        {'embedding_dim': 12, 'use_user_bias': False, 'use_item_bias': True, 'use_global_bias': False}, DS())
    assert m2.embedding_dim == 12 and m2.use_item_bias
    loss = RecommenderSystemLossesEnum['sampled_softmax'].value.build_from_conf(
        {'train_neg_strategy': 'uniform', 'neg_train': 10}, DS())
    assert abs(loss.neg_shift() - np.log(120 / 10)) < 1e-12


def test_synthetic_data_is_seeded_and_split_disjoint():
    from hassaku_b200.data.synthetic import make_interactions
    a = make_interactions(300, 200, 6000, seed=0, n_user_groups=2)
    b = make_interactions(300, 200, 6000, seed=0, n_user_groups=2)
    assert (a.train != b.train).nnz == 0 and (a.val != b.val).nnz == 0
    assert a.train.multiply(a.val).nnz == 0 and a.train.multiply(a.test).nnz == 0 and a.val.multiply(a.test).nnz == 0
    n = a.train.nnz + a.val.nnz + a.test.nnz
    assert 0.75 < a.train.nnz / n < 0.85
    assert a.train.has_sorted_indices


def test_datasets_from_csv_equal_from_interactions():
    from hassaku_b200.data.dataset import FullEvalDataset, TrainRecDataset
    from hassaku_b200.data.synthetic import make_interactions, write_csv_dataset
    data = make_interactions(60, 150, 1500, seed=1, n_user_groups=2)
    with tempfile.TemporaryDirectory() as tmp:
        write_csv_dataset(data, tmp)
        t1 = TrainRecDataset(tmp)
        e1 = FullEvalDataset(tmp, 'test')
    t2 = TrainRecDataset.from_interactions(data.train, data.user_group, 2)
    e2 = FullEvalDataset.from_interactions(data.test, data.train + data.val, 'test', data.user_group, 2)
    assert (t1.sampling_matrix != t2.sampling_matrix).nnz == 0 and len(t1) == len(t2) == data.train.nnz
    assert (e1.iteration_matrix != e2.iteration_matrix).nnz == 0
    assert (e1.exclude_data.astype(bool) != e2.exclude_data.astype(bool)).nnz == 0
    assert e1.n_user_groups == e2.n_user_groups == 2
    assert torch.equal(e1.user_to_user_group, e2.user_to_user_group)
    u, items, y = e1[5]
    assert items.shape == (150,) and y.dtype == np.float32 and y.sum() == data.test[5].nnz
    uu, ii, one = t1[0]
    assert data.train[uu, ii] == 1 and one == 1.
    np.testing.assert_allclose(t1.pop_distribution.sum(), 1.0)


def test_bench_batches_follow_loader_semantics_and_byte_accounting():
    import bench
    from hassaku_b200.data.synthetic import make_interactions
    data = make_interactions(300, 200, 6000, seed=0)
    us, its = bench.make_batches(data, 64, 20, 3)
    for u, i in zip(us, its):
        assert u.dtype == np.int64 and i.shape == (64, 21)
        for r in range(64):
            row = data.train[u[r]].indices
            assert i[r, 0] in row and not np.isin(i[r, 1:], row).any()
    # BASELINE.md §3 byte table
    assert abs(bench.algorithmic_bytes(6040, 3706, 402, 128, 50)['total'] / 1e6 - 131.3) < 0.1
    assert abs(bench.algorithmic_bytes(6040, 3706, 402, 8192, 50)['total'] / 1e6 - 1486.5) < 0.1
    assert abs(bench.algorithmic_bytes(69878, 10677, 128, 8192, 100)['total'] / 1e6 - 1157.9) < 0.1


def test_header_is_plain_c_and_a_c_host_links(tmp_path):
    """The drop-in boundary is a C ABI: include/hassaku_b200.h compiles as C99 (-pedantic) and as C++11, and a C program
    links against the library and calls its CUDA-free entry points (examples/c_abi_link_check.c)."""
    import shutil
    import subprocess
    if shutil.which('gcc') is None:
        pytest.skip('gcc not available')
    from hsk_testutil import ROOT
    inc, libdir = os.path.join(ROOT, 'include'), os.path.join(ROOT, 'hassaku_b200', 'lib')
    src = os.path.join(ROOT, 'examples', 'c_abi_link_check.c')
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror', '-I', inc, '-fsyntax-only', src], check=True)
    subprocess.run(['g++', '-std=c++11', '-Wall', '-Wextra', '-Werror', '-I', inc, '-fsyntax-only', '-x', 'c++', src], check=True)
    exe = str(tmp_path / 'c_abi_check')
    subprocess.run(['gcc', '-std=c99', '-I', inc, src, '-L', libdir, '-lhassaku_b200', f'-Wl,-rpath,{libdir}', '-o', exe],
                   check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert 'hsk_version' in out and 'tables are null' in out
    # the ctypes mirrors have the layout the C compiler gives the header's structs
    import ctypes
    import re
    from hassaku_b200 import _C
    sizes = dict((k, int(v)) for k, v in re.findall(r'(hsk_\w+)=(\d+)', out))
    assert sizes == {'hsk_mf_tables': ctypes.sizeof(_C.MfTables), 'hsk_row_segment': ctypes.sizeof(_C.RowSegment),
                     'hsk_peer_items': ctypes.sizeof(_C.PeerItems), 'hsk_peer_flags': ctypes.sizeof(_C.PeerFlags)}, sizes


def test_item_shards_and_peer_tables_host_side():
    """The ctypes side of the shard / peer entry points (no GPU): array layout, limits, null handling."""
    import ctypes
    from hassaku_b200 import _C
    sh = _C.ItemShards([10, 9, 9], Vq=[0x1000, 0x2000, 0x3000], V=[0x10, 0x20, 0x30])
    assert sh.n == 3 and list(sh.rows) == [10, 9, 9] and sh.Ib is None and sh.Vq[1] == 0x2000
    with pytest.raises(ValueError):
        _C.ItemShards(list(range(1, 10)))                       # more than HSK_MAX_PEERS shards
    p = _C.make_peer_items([1, 2], [3, 4])
    assert p.world == 2 and p.V[1] == 2 and p.gV[0] == 3 and not p.Ib[0] and not p.stamps[1]
    with pytest.raises(ValueError):
        _C.make_peer_items(list(range(9)), list(range(9)))
    f = _C.make_peer_flags([16, 32, 48], 2)
    assert (f.world, f.rank, f.flags[2]) == (3, 2, 48)
    # scratch sizing of the shard evaluator is CUDA-free except for the SM count: monotone in the batch
    assert ctypes.sizeof(_C.PeerItems) == 8 + 5 * 8 * _C.MAX_PEERS


def test_step_entry_points_take_an_empty_batch_without_index_pointers():
    """A rank whose share of the global batch is empty passes empty index tensors, and torch gives an empty tensor a null data
    pointer: the step entry points accept B = 0 without indices (and launch nothing); B > 0 still needs them."""
    import ctypes
    from hassaku_b200 import _C
    lib = _C.lib()
    t = _C.MfTables(0x1000, 0x2000, None, None, None, 4, 4, 4, 4)
    g = _C.MfTables(0x3000, 0x4000, None, None, None, 4, 4, 4, 4)
    p = _C.make_peer_items([0x2000, 0x5000], [0x4000, 0x6000])
    for B, rc in ((0, 0), (3, -1)):
        assert lib.hsk_mf_train_fused_v(ctypes.byref(t), ctypes.byref(g), None, None, B, 6, 8, 0, 0.0, None, None, None,
                                        None, 0, None) == rc
        assert lib.hsk_mf_train_fused_peer(ctypes.byref(t), ctypes.byref(g), ctypes.byref(p), None, None, B, 6, 8, 0, 0.0, None,
                                           1, None, None, None) == rc
    assert b'null' in lib.hsk_last_error()
