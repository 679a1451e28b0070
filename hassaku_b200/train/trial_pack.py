"""Trial packs: M SGDMatrixFactorization models of ONE shape (a hyperparameter sweep) trained in one process, with one
fused-step launch and one optimizer launch per step for all of them.

The models share the dataset, embedding_dim, bias flags, loss, neg_train, batch size and optimizer, and differ in lr,
weight decay, initial weights (init seed), n_epochs and patience.  Their parameter arenas become the rows of one
[M, stride] fp32 allocation (stride = the single-model ArenaLayout.n_total, a multiple of 32 elements, so every table keeps
its 128-byte alignment); m, v and the gradient arena are laid out the same way.  Each model is rebound to its row
(`_set_arena`), so `state_dict()`, `save_model_to_path`, `forward` and the evaluator work on it unchanged.

A step (`PackedMFTrainStep.step`) enqueues hsk_mf_train_fused_pack, hsk_mark_batch and hsk_adamw_pack for the active
trials; the per-trial AdamW scalars of a whole epoch are computed on the host once (hsk_adamw_consts_table) and uploaded in
one copy.  Under torch.use_deterministic_algorithms(True) each active trial instead runs the single-model deterministic
step (hsk_mf_train_fused_det) and its own AdamW on its row of the pack: slower, but every trial gives the same bits as
its own `Trainer`.

Shared batches, deliberately: every trial of a pack sees the loader's batch sequence.  A trial that trains k epochs in a
pack therefore sees exactly the batches that a `Trainer` with a fresh loader of the same seed sees in its k epochs; trials
that stop early simply stop consuming them.

`PackedTrainer` is `Trainer.fit` for the M trials over one shared loader: per trial the initial validation, early stopping
on its own `optimizing_metric` / `max_patience` / `n_epochs`, a checkpoint to its `model_path` on every improvement, the
same prints and the same returned dict.  A trial that runs out of patience or epochs is deactivated at that epoch boundary.
The initial validation and each epoch's validation are one packed sweep over the trials concerned (evaluate_mf_pack:
one top-k and one metrics launch per chunk of users for all of them); models with a tensor-core `eval_precision` are
validated one by one instead.

Packing pays where one trial's step is launch-bound (measured on a B200 at the ML-1M shape: up to 11.6x at B 64, d 64;
2.1x at d 402, where the pack's AdamW pass runs at HBM bandwidth).  It does not pay for bpr / bce with d > 96 at large
batches (0.82x at B 8192 x 50, d 402): the single-model step uses the bulk-copy ring kernel there, which is not packed
(DESIGN.md section 10).

    from collections import defaultdict
    packs = defaultdict(list)
    for conf in sweep_confs:
        packs[shape_key(conf)].append(conf)
"""
import torch

from hassaku_b200 import _C, determinism
from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
from hassaku_b200.eval.eval import FullEvaluator, evaluate_mf_pack, evaluate_recommender_algorithm
from hassaku_b200.train.optim import stamp_segments
from hassaku_b200.train.rec_losses import RecommenderSystemLoss
from hassaku_b200.train.trainer_step import HostBatchStager

# conf keys that must agree within a pack: they fix the tensors' shapes, the batches or the optimizer
SHAPE_KEYS = ('dataset_path', 'embedding_dim', 'use_user_bias', 'use_item_bias', 'use_global_bias', 'rec_loss', 'neg_train',
              'train_neg_strategy', 'train_batch_size', 'optimizer', 'optimizer_mode', 'device')
_OPTIMIZERS = {'adamw': False, 'adam': True}   # name -> Adam(L2)?
_MISSING = object()


def shape_key(conf: dict) -> tuple:
    """The part of a trial configuration that must be equal across one pack (group a sweep's confs by it)."""
    return tuple((k, repr(conf.get(k))) for k in SHAPE_KEYS)


def _model_key(model) -> dict:
    return {'n_users': model.n_users, 'n_items': model.n_items, 'embedding_dim': model.embedding_dim,
            'use_user_bias': model.use_user_bias, 'use_item_bias': model.use_item_bias,
            'use_global_bias': model.use_global_bias}


def _check_models(models):
    if not models:
        raise ValueError('a trial pack needs at least one model')
    for m in models:
        if not isinstance(m, SGDMatrixFactorization):
            raise TypeError('a trial pack trains hassaku_b200 SGDMatrixFactorization models only')
    ref = _model_key(models[0])
    for j, m in enumerate(models[1:], 1):
        for k, v in _model_key(m).items():
            if ref[k] != v:
                raise ValueError(f"model {j} differs from model 0 in '{k}' ({v} vs {ref[k]}): one pack holds models of one shape")


def _check_single_process():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        raise ValueError(f'trial packs are single-GPU: the process group has {dist.get_world_size()} ranks '
                         f"(key 'multi_gpu': run one pack per rank)")


class PackedMFTrainStep:
    """One training step of M models of one shape: the fused step and AdamW / Adam(L2) of every active trial in one launch
    each.  `lrs` / `wds`: one learning rate / weight decay per model; `optimizer`: 'adamw' or 'adam'."""

    def __init__(self, models, rec_loss: RecommenderSystemLoss, lrs, wds, optimizer: str = 'adamw', betas=(0.9, 0.999),
                 eps: float = 1e-8):
        _check_models(models)
        _check_single_process()
        if optimizer not in _OPTIMIZERS:
            raise ValueError(f"optimizer '{optimizer}' has no packed implementation (adamw, adam)")
        if rec_loss.loss_kind not in _C.LOSS_KINDS:
            raise ValueError(f'Loss {rec_loss.name} has no fused kernel')
        M = len(models)
        if len(lrs) != M or len(wds) != M:
            raise ValueError(f'one lr and one wd per model: {M} models, {len(lrs)} lrs, {len(wds)} wds')
        for wd in wds:
            # the kernel applies weight decay when its fp32 copy is non-zero; torch tests the double
            if wd != 0.0 and float(torch.tensor(wd, dtype=torch.float32)) == 0.0:
                raise ValueError(f"weight decay 'wd' = {wd} rounds to 0 in fp32")
        self.device = models[0].arena.device
        if self.device.type != 'cuda':
            raise ValueError("trial packs need the models on a CUDA device (key 'device': cuda); there is no CPU path")
        self.models, self.rec_loss = list(models), rec_loss
        self.lrs, self.wds = [float(x) for x in lrs], [float(x) for x in wds]
        self.adam_l2 = _OPTIMIZERS[optimizer]
        self.betas, self.eps = (float(betas[0]), float(betas[1])), float(eps)
        self.kind = _C.LOSS_KINDS[rec_loss.loss_kind]
        self.shift = float(rec_loss.neg_shift())
        self.layout = lay = models[0].layout
        self.stride = lay.n_total
        need = M * 4 * self.stride * 4
        free, _total = torch.cuda.mem_get_info(self.device)
        if need > free:
            raise _C.HskError(f'a pack of {M} trials needs {need / 2**30:.2f} GiB for parameters, m, v and gradients '
                              f'({M} x 4 x {self.stride} fp32); {free / 2**30:.2f} GiB of {self.device} are free: '
                              f'split the sweep into smaller packs')
        self.p = torch.empty((M, self.stride), dtype=torch.float32, device=self.device)
        for j, m in enumerate(self.models):
            self.p[j].copy_(m.arena.detach())
            m._set_arena(self.p[j])
        self.m = torch.zeros_like(self.p)
        self.v = torch.zeros_like(self.p)
        self.g = torch.zeros_like(self.p)
        self.tables = lay.tables(self.p[0])
        self.grad_tables = lay.tables(self.g[0])
        self.stamp_users = torch.zeros(lay.n_users, dtype=torch.uint8, device=self.device)
        self.stamp_items = torch.zeros(lay.n_items, dtype=torch.uint8, device=self.device)
        self.loss_accum = torch.zeros(M, dtype=torch.float64, device=self.device)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.t = 0                        # optimizer steps taken (every active trial has taken the same number)
        self._consts, self._consts_t0 = None, 1
        self._stager = HostBatchStager(self.device)
        self.set_active([True] * M)

    @property
    def n_trials(self) -> int:
        return len(self.models)

    def set_active(self, mask):
        """Select the trials the following steps train (call at epoch boundaries); `mask`: one bool per trial."""
        if len(mask) != self.n_trials:
            raise ValueError(f'set_active: {len(mask)} flags for {self.n_trials} trials')
        self.active_idx = [j for j, a in enumerate(mask) if a]
        self.active = torch.tensor(self.active_idx or [0], dtype=torch.int32).to(self.device)[:len(self.active_idx)]

    def prepare(self, n_steps: int):
        """Compute the AdamW scalars of every trial for the next `n_steps` steps and upload them in one copy (the
        trainer calls it with the epoch's batch count; `step` extends the table itself when it runs past the end)."""
        n_steps = max(int(n_steps), 1)
        host = _C.adamw_consts_table(self.lrs, self.wds, self.betas[0], self.betas[1], self.eps, self.t + 1, n_steps,
                                     torch.empty((n_steps, self.n_trials, 8), dtype=torch.float32, pin_memory=True))
        self._consts = host.to(self.device, non_blocking=True)
        self._consts_t0 = self.t + 1

    def step(self, u_idxs: torch.Tensor, i_idxs: torch.Tensor):
        """Enqueue one step of every active trial on the batch (u_idxs [B], i_idxs [B, 1 + N]; host or device)."""
        if not self.active_idx:
            return
        slot, u, i = self._stager.device_batch(u_idxs, i_idxs)
        segs, su, si = stamp_segments(self.layout, int(u.numel()), int(i.numel()), self.stamp_users, self.stamp_items)
        if determinism.enabled():
            self._step_deterministic(u, i, segs, su, si)
        else:
            k = self.t + 1 - self._consts_t0
            if self._consts is None or k >= self._consts.shape[0]:
                self.prepare(64)
                k = 0
            _C.mf_train_fused_pack(self.tables, self.grad_tables, self.stride, self.n_trials, self.active, u, i, self.kind,
                                   self.shift, self.loss_accum, status=self.status)
            if segs:
                _C.mark_batch(u, i, self.layout.n_users, self.layout.n_items, su, si, step=self.t + 1)
            self.t += 1
            _C.adamw_pack(self.p, self.m, self.v, self.g, self.active, self._consts[k], segs, step=self.t,
                          adam_l2=self.adam_l2, status=self.status)
        if slot is not None:
            slot['free'].record()

    def _step_deterministic(self, u, i, segs, su, si):
        """Each active trial through the single-model deterministic step and its own optimizer call: the same launches,
        on the same data, as that trial's `Trainer` (FusedMFTrainStep + DenseAdam)."""
        lay = self.layout
        scratch = determinism.scratch(self, _C.det_scratch_bytes(i.shape[0], i.shape[1], lay.ld), self.device)
        for j in self.active_idx:
            _C.mf_train_fused_det(self.models[j]._tables(), lay.tables(self.g[j]), u, i, self.kind, self.shift,
                                  self.loss_accum[j:j + 1], scratch, status=self.status)
        if segs:
            _C.mark_batch(u, i, lay.n_users, lay.n_items, su, si, step=self.t + 1)
        self.t += 1
        b1, b2 = self.betas
        for j in self.active_idx:
            if segs:
                _C.adamw_dense_rows(self.p[j], self.m[j], self.v[j], self.g[j], segs, self.lrs[j], b1, b2, self.eps,
                                    self.wds[j], self.t, arith=0, adam_l2=self.adam_l2)
            else:
                _C.adamw_dense(self.p[j], self.m[j], self.v[j], self.g[j], self.lrs[j], b1, b2, self.eps, self.wds[j], self.t,
                               arith=0, adam_l2=self.adam_l2, zero_grad=True)

    def check_status(self):
        """Host sync: IndexError if a kernel met an out-of-range user, item or trial index since the last check."""
        st = int(self.status.item())
        if st & _C.STATUS_BAD_INDEX:
            self.status.zero_()
            raise IndexError('index out of range in a trial pack (user, item or active-trial index)')

    def pop_loss_sums(self):
        """One host sync: per trial, the sum of its batch-mean losses since the last call (list of M floats)."""
        v = self.loss_accum.tolist()
        self.loss_accum.zero_()
        self.check_status()
        return v


def _check_conf(j: int, conf: dict):
    dev = str(conf.get('device', 'cpu'))
    if not dev.startswith('cuda'):
        raise ValueError(f"conf {j}: 'device' is {dev!r}: trial packs run on a CUDA device only")
    if conf.get('optimizer') not in _OPTIMIZERS:
        raise ValueError(f"conf {j}: 'optimizer' {conf.get('optimizer')!r} has no packed implementation (adamw, adam)")
    if conf.get('optimizer_mode', 'dense') != 'dense':
        raise ValueError(f"conf {j}: 'optimizer_mode' {conf.get('optimizer_mode')!r}: trial packs use the dense optimizer")
    if conf.get('running_settings', {}).get('use_wandb', False):
        raise ValueError(f"conf {j}: 'use_wandb' is set: trial packs do not report to W&B")
    if conf.get('_in_tune', False):
        raise ValueError(f"conf {j}: '_in_tune' is set: trial packs do not report to Ray Tune")


def check_confs(confs):
    """Reject what a pack cannot run, naming the offending key: a shape key that differs between confs, adagrad, lazy
    AdamW, W&B / Ray Tune reporting, a CPU device."""
    if not confs:
        raise ValueError('a trial pack needs at least one conf')
    for j, c in enumerate(confs):
        _check_conf(j, c)
    for k in SHAPE_KEYS:
        v0 = confs[0].get(k, _MISSING)
        for j, c in enumerate(confs[1:], 1):
            v = c.get(k, _MISSING)
            if v != v0:
                raise ValueError(f"conf {j} differs from conf 0 in shape key '{k}' ({None if v is _MISSING else v!r} vs "
                                 f"{None if v0 is _MISSING else v0!r}): group a sweep into packs by shape_key(conf)")


class TrialSchedule:
    """Early stopping of `Trainer.fit`, per trial, as host logic: validation before any update, then per epoch the
    patience / n_epochs test at the epoch's start, the train epoch and the validation."""

    def __init__(self, n_epochs, max_patience):
        self.n_epochs, self.max_patience = list(n_epochs), list(max_patience)
        M = len(self.n_epochs)
        self.patience = list(self.max_patience)
        self.done = [False] * M
        self.best_value = [None] * M
        self.best_epoch = [None] * M
        self.best_metrics = [None] * M
        self.epoch = 0

    def start(self, j: int, value, metrics: dict):
        self.best_value[j] = metrics['max_optimizing_metric'] = value
        self.best_epoch[j] = metrics['best_epoch'] = -1
        self.best_metrics[j] = metrics

    def begin_epoch(self):
        """Trials that train this epoch; a trial out of epochs or patience is done from here on.  Returns (active trial
        indices, trials that ran out of patience at this boundary)."""
        active, stopped = [], []
        for j in range(len(self.done)):
            if self.done[j]:
                continue
            if self.epoch >= self.n_epochs[j]:
                self.done[j] = True
            elif self.patience[j] == 0:
                self.done[j] = True
                stopped.append(j)
            else:
                active.append(j)
        return active, stopped

    def end_epoch(self, j: int, value, metrics: dict) -> bool:
        """Record trial j's validation of the current epoch; True when it is a new best (checkpoint)."""
        if value > self.best_value[j]:
            self.best_value[j], self.best_epoch[j], self.best_metrics[j] = value, self.epoch, metrics
            metrics['max_optimizing_metric'], metrics['best_epoch'] = value, self.epoch
            self.patience[j] = self.max_patience[j]
            return True
        metrics['max_optimizing_metric'] = self.best_value[j]
        self.patience[j] -= 1
        return False


class PackedTrainer:
    """`Trainer.fit` for M trials of one shape over one shared loader.  `models[j]` is built from `confs[j]`
    (SGDMatrixFactorization.build_from_conf after seeding trial j's init); `fit()` returns the `best_metrics` of every
    trial, in the order of `confs`."""

    def __init__(self, models, train_loader, val_loader, rec_loss: RecommenderSystemLoss, confs):
        confs = list(confs)
        if len(models) != len(confs):
            raise ValueError(f'one conf per model: {len(models)} models, {len(confs)} confs')
        check_confs(confs)
        _check_models(models)
        _check_single_process()
        self.confs = confs
        self.device = confs[0]['device']
        for m in models:
            m.to(self.device)
        self.models = list(models)
        self.train_loader, self.val_loader, self.rec_loss = train_loader, val_loader, rec_loss
        self.batch_verbose = confs[0].get('running_settings', {}).get('batch_verbose', False)
        self.train_step = PackedMFTrainStep(self.models, rec_loss, [c['lr'] for c in confs], [c['wd'] for c in confs],
                                            optimizer=confs[0]['optimizer'])
        self.schedule = TrialSchedule([c['n_epochs'] for c in confs], [c['max_patience'] for c in confs])
        self.epoch_losses = [[] for _ in confs]    # per trial, the dicts of its train epochs

    def _evaluator(self) -> FullEvaluator:
        ds = self.val_loader.dataset
        return FullEvaluator(aggr_by_group=True, n_groups=ds.n_user_groups, user_to_user_group=ds.user_to_user_group)

    @torch.no_grad()
    def val(self, j: int) -> dict:
        """Trainer.val for trial j: full-rank evaluation on the validation loader -> metric dict."""
        model = self.models[j]
        model.eval()
        print('Validation started')
        return evaluate_recommender_algorithm(model, self.val_loader, self._evaluator(), self.device, self.batch_verbose)

    @torch.no_grad()
    def val_pack(self, trials) -> dict:
        """Trainer.val for every trial of `trials` in one packed sweep -> {trial: metric dict}; {} when a model evaluates
        in a tensor-core precision (evaluate_mf_pack runs the fp32 evaluator only: such packs use `val` per trial)."""
        if any(getattr(m, 'eval_precision', 'fp32') != 'fp32' for m in self.models):
            return {}
        for j in trials:
            self.models[j].eval()
        res = evaluate_mf_pack([self.models[j] for j in trials], self.val_loader, [self._evaluator() for _ in trials],
                               self.device, self.batch_verbose)
        return dict(zip(trials, res))

    def _val_result(self, j: int, packed: dict) -> dict:
        """Trial j's validation: its entry of the packed sweep (with val's print), or `val(j)`."""
        if j not in packed:
            return self.val(j)
        print('Validation started')
        return packed[j]

    def _train_one_epoch(self, active) -> dict:
        for j in active:
            self.models[j].train()
        n_batches = 0
        for u_idxs, i_idxs, _labels in self.train_loader:
            self.train_step.step(u_idxs, i_idxs)
            n_batches += 1
        sums = self.train_step.pop_loss_sums()     # the only host sync of the epoch
        out = {}
        for j in active:
            rec = sums[j] / max(n_batches, 1)
            out[j] = {'epoch_train_loss': rec, 'epoch_train_rec_loss': rec, 'epoch_train_reg_loss': 0.0}
        return out

    def fit(self):
        sch = self.schedule
        packed = self.val_pack(list(range(len(self.confs))))
        for j, conf in enumerate(self.confs):
            first = self._val_result(j, packed)
            sch.start(j, first[conf['optimizing_metric']], first)
            print('Init - Avg Val Value {:.3f} \n'.format(sch.best_value[j]))
            self.models[j].save_model_to_path(conf['model_path'])
        while True:
            active, stopped = sch.begin_epoch()
            for _ in stopped:
                print('Ran out of patience, Stopping ')
            if not active:
                break
            self.train_step.set_active([j in active for j in range(len(self.confs))])
            self.train_step.prepare(len(self.train_loader))
            losses = self._train_one_epoch(active)
            packed = self.val_pack(active)
            epoch = sch.epoch
            for j in active:
                lj = losses[j]
                self.epoch_losses[j].append(lj)
                print('Epoch {} - Epoch Avg Train Loss {:.4f} ({:.4f} Rec Loss + {:.4f} Reg Loss )\n'.format(
                    epoch, lj['epoch_train_loss'], lj['epoch_train_rec_loss'], lj['epoch_train_reg_loss']))
                metrics = self._val_result(j, packed)
                value = metrics[self.confs[j]['optimizing_metric']]
                print('Epoch {} - Avg Val Value {:.4f} \n'.format(epoch, value))
                if sch.end_epoch(j, value, metrics):
                    print('Epoch {} - New best model found (val value {:.4f}) \n'.format(epoch, value))
                    self.models[j].save_model_to_path(self.confs[j]['model_path'])
            sch.epoch += 1
        return list(sch.best_metrics)
