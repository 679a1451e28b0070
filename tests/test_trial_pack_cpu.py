"""CPU tests of the trial pack's host side: conf / shape-key validation and every rejected option, the per-epoch AdamW
constants table against hsk_adamw_consts, argument checks of the new entry points, and the early-stopping schedule."""
import ctypes

import numpy as np
import pytest
import torch


def _conf(**kw):
    c = {'device': 'cuda', 'lr': 1e-3, 'wd': 0.0, 'optimizer': 'adamw', 'n_epochs': 3, 'optimizing_metric': 'ndcg@10',
         'max_patience': 2, 'model_path': '/nonexistent', 'embedding_dim': 64, 'neg_train': 4, 'train_batch_size': 64,
         'running_settings': {'use_wandb': False, 'batch_verbose': False}}
    c.update(kw)
    return c


@pytest.mark.parametrize('bad,key', [
    ({'device': 'cpu'}, 'device'),
    ({'optimizer': 'adagrad'}, 'optimizer'),
    ({'optimizer_mode': 'lazy'}, 'optimizer_mode'),
    ({'running_settings': {'use_wandb': True, 'batch_verbose': False}}, 'use_wandb'),
    ({'_in_tune': True}, '_in_tune'),
])
def test_rejected_options_name_their_key(bad, key):
    from hassaku_b200.train.trial_pack import check_confs
    with pytest.raises(ValueError, match=f"'{key}'"):
        check_confs([_conf(), _conf(**bad)])


@pytest.mark.parametrize('key,val', [('embedding_dim', 32), ('neg_train', 10), ('train_batch_size', 1024),
                                     ('optimizer', 'adam'), ('use_item_bias', True), ('rec_loss', 'bce')])
def test_shape_key_mismatch_names_the_key(key, val):
    from hassaku_b200.train.trial_pack import check_confs, shape_key
    a, b = _conf(), _conf(**{key: val})
    assert shape_key(a) != shape_key(b)
    with pytest.raises(ValueError, match=f"'{key}'"):
        check_confs([a, b])


def test_confs_differing_in_trial_keys_form_one_pack():
    from hassaku_b200.train.trial_pack import check_confs, shape_key
    confs = [_conf(lr=1e-3, wd=0.0, n_epochs=5, max_patience=1, model_path='/a'),
             _conf(lr=3e-4, wd=1e-4, n_epochs=2, max_patience=3, model_path='/b', optimizing_metric='recall@20')]
    check_confs(confs)
    assert shape_key(confs[0]) == shape_key(confs[1])


def test_models_of_another_shape_are_rejected():
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.trial_pack import _check_models
    a = SGDMatrixFactorization(30, 20, 8)
    with pytest.raises(ValueError, match="'embedding_dim'"):
        _check_models([a, SGDMatrixFactorization(30, 20, 16)])
    with pytest.raises(ValueError, match="'use_item_bias'"):
        _check_models([a, SGDMatrixFactorization(30, 20, 8, use_item_bias=True)])
    with pytest.raises(ValueError, match="'n_items'"):
        _check_models([a, SGDMatrixFactorization(30, 21, 8)])
    _check_models([a, SGDMatrixFactorization(30, 20, 8)])


def test_cpu_models_are_rejected():
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trial_pack import PackedMFTrainStep
    with pytest.raises(ValueError, match="'device'"):
        PackedMFTrainStep([SGDMatrixFactorization(30, 20, 8)], RecBayesianPersonalizedRankingLoss(), [1e-3], [0.0])


def test_multi_rank_process_group_is_rejected(monkeypatch):
    import torch.distributed as dist
    from hassaku_b200.train import trial_pack
    monkeypatch.setattr(dist, 'is_initialized', lambda: True)
    monkeypatch.setattr(dist, 'get_world_size', lambda *a, **k: 2)
    with pytest.raises(ValueError, match='ranks'):
        trial_pack._check_single_process()


def test_constants_table_equals_hsk_adamw_consts():
    from hassaku_b200 import _C
    lrs, wds = [1e-3, 3e-4, 5e-2, 1e-3], [0.0, 4e-5, 1e-2, 0.0]
    b1, b2, eps, first, n = 0.9, 0.999, 1e-8, 7, 40
    tab = _C.adamw_consts_table(lrs, wds, b1, b2, eps, first, n)
    assert tab.shape == (n, len(lrs), 8)
    one = torch.empty(8, dtype=torch.float32)
    for s in range(n):
        for j in range(len(lrs)):
            _C.adamw_consts(lrs[j], b1, b2, eps, wds[j], first + s, one)
            assert torch.equal(tab[s, j].view(torch.int32), one.view(torch.int32)), (s, j)
    assert float(tab[:, 0, 1].abs().max()) == 0.0 and float(tab[:, 3, 1].abs().max()) == 0.0   # wd = 0 trials


def test_pack_entry_points_validate_without_gpu():
    from hassaku_b200 import _C
    lib = _C.lib()
    t = _C.MfTables(16, 4096, None, None, None, 10, 10, 4, 4)     # fake, aligned: validation fails before any launch
    g = _C.MfTables(8192, 12288, None, None, None, 10, 10, 4, 4)
    act = 64
    for stride, n_trials, n_active, what in ((6, 2, 1, b'trial_stride'), (0, 2, 1, b'trial_stride'),
                                             (88, 2, 3, b'n_active'), (88, 0, 0, b'n_trials')):
        rc = lib.hsk_mf_train_fused_pack(ctypes.byref(t), ctypes.byref(g), stride, n_trials, act, n_active, 32, 48, 4, 3, 0, 0.0,
                                         None, None, None)
        assert rc == -1 and what in lib.hsk_last_error(), (stride, n_trials, n_active, lib.hsk_last_error())
    rc = lib.hsk_mf_train_fused_pack(ctypes.byref(t), ctypes.byref(g), 88, 2, None, 1, 32, 48, 4, 3, 0, 0.0, None, None, None)
    assert rc == -1 and b'active' in lib.hsk_last_error()
    rc = lib.hsk_adamw_pack(None, None, None, None, 88, 2, act, 1, 16, None, 0, 1, 0, None, None)
    assert rc == -1 and b'null' in lib.hsk_last_error()
    rc = lib.hsk_adamw_pack(16, 32, 48, 64, 88, 2, act, 1, 8, None, 0, 1, 0, None, None)
    assert rc == -1 and b'aligned' in lib.hsk_last_error()
    rc = lib.hsk_adamw_pack(16, 32, 48, 64, 90, 2, act, 1, 16, None, 0, 1, 0, None, None)
    assert rc == -1 and b'trial_stride' in lib.hsk_last_error()
    seg = (_C.RowSegment * 1)(_C.RowSegment(80, 4, 4, 256))      # runs past the trial's row
    rc = lib.hsk_adamw_pack(16, 32, 48, 64, 88, 2, act, 1, 16, seg, 1, 1, 0, None, None)
    assert rc == -1 and b'segment' in lib.hsk_last_error()


def _trainer_fit_schedule(values, n_epochs, max_patience):
    """Trainer.fit's control flow (train/trainer.py) for one trial, on a scripted metric sequence: (epochs trained,
    best epoch, best value, number of 'Ran out of patience' prints)."""
    best, best_epoch, patience, trained, stops = values[0], -1, max_patience, 0, 0
    for epoch in range(n_epochs):
        if patience == 0:
            stops += 1
            break
        trained += 1
        v = values[1 + epoch]
        if v > best:
            best, best_epoch, patience = v, epoch, max_patience
        else:
            patience -= 1
    return trained, best_epoch, best, stops


def test_early_stopping_schedule_matches_trainer_per_trial():
    from hassaku_b200.train.trial_pack import TrialSchedule
    rng = np.random.RandomState(0)
    M = 6
    n_epochs = [1, 4, 6, 3, 8, 5]
    max_pat = [1, 1, 2, 5, 1, 3]
    values = [list(np.round(rng.rand(1 + 8), 1)) for _ in range(M)]   # ties are frequent: "not better" keeps patience going down
    values[4] = [0.5, 0.5, 0.5, 0.9, 0.9]                               # patience 1: stops after one epoch without improvement
    sch = TrialSchedule(n_epochs, max_pat)
    for j in range(M):
        sch.start(j, values[j][0], {})
    trained, stops, active_sets = [0] * M, [0] * M, []
    while True:
        active, stopped = sch.begin_epoch()
        for j in stopped:
            stops[j] += 1
        if not active:
            break
        active_sets.append(active)
        for j in active:
            trained[j] += 1
            sch.end_epoch(j, values[j][1 + sch.epoch], {})
        sch.epoch += 1
    for j in range(M):
        want = _trainer_fit_schedule(values[j], n_epochs[j], max_pat[j])
        assert (trained[j], sch.best_epoch[j], sch.best_value[j], stops[j]) == want, j
    # a trial, once inactive, never comes back
    for e in range(1, len(active_sets)):
        assert set(active_sets[e]) <= set(active_sets[e - 1])
    assert trained[4] == 1 and stops[4] == 1
