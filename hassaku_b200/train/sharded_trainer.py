"""Multi-GPU `Trainer.fit()` for SGDMatrixFactorization: what `nn.DataParallel(self.model)` does in the reference
(train/trainer.py:38-40), re-designed for one process per GPU.

Launch with torchrun (one rank per GPU); EVERY rank builds the same model / datasets / conf exactly as for the single-GPU
`Trainer` and calls `ShardedTrainer(model, train_loader, val_loader, rec_loss, conf).fit()`:

  * the tables are row-sharded (user u and item i live on rank u % G / i % G: hassaku_b200/sharded.py), so per-GPU memory and
    the optimizer pass shrink with G — DataParallel replicates the model and reduces dense gradients on GPU 0;
  * a rank trains on the interactions of ITS users: a device-resident loader over that slice (device shuffle +
    hsk_sample_negatives); `train_batch_size` is the GLOBAL batch like DataParallel's (each rank takes 1 / G of it), the
    loss normalisers stay global, so a step is the single-GPU step on the union batch;
  * the item rows a rank needs are read from / their gradients reduced into the owners' memory by the step kernel over
    NVLink (`exchange='peer'`, one node, rows <= 128 floats) or exchanged by NCCL all-to-all (`'sparse'`) / all-gather +
    reduce-scatter (`'dense'`, batches that cover the item table) — chosen per shape unless `conf['sharded_exchange']` says
    otherwise; `'ordered'` is the sparse exchange with every float reduction in a fixed order: with it, fit() under
    torch.use_deterministic_algorithms(True) gives the same checkpoint, metrics and losses on every run at a fixed world size;
  * validation is the sharded full-rank evaluator (`ShardedMF.evaluate_replicated` while the item table fits one GPU, the
    item-sharded protocol otherwise): every rank gets the same metric dict, so early stopping needs no extra collective;
  * the best model is written by rank 0 as the reference's `model.pth` (full state_dict, reference key names / shapes).

Same control flow, conf keys, printed lines and returned dict as `Trainer.fit` (train/trainer.py:85-185).  The loss per
epoch is the mean over the steps of the batch-mean loss, as there.  An epoch has floor(min over ranks(local interactions) /
local batch) steps (fixed shapes: the step is replayed as one CUDA graph); the few tail interactions of an epoch are
dropped, a different random subset each epoch.
"""
import logging
import os

import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

from hassaku_b200 import _C
from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
from hassaku_b200.data.dataloader import NegativeSampler, TrainDataLoader
from hassaku_b200.data.dataset import TrainRecDataset
from hassaku_b200.eval.eval import FullEvaluator
from hassaku_b200.sharded import ShardedMF

MODEL_FILE = 'model.pth'


class ShardedTrainer:
    EXCHANGES = ('auto', 'peer', 'sparse', 'dense', 'ordered')

    def __init__(self, model: SGDMatrixFactorization, train_loader, val_loader, rec_loss, conf: dict, group=None):
        if not dist.is_initialized():
            raise _C.HskError('ShardedTrainer needs torch.distributed (launch with torchrun, one rank per GPU); '
                              'single GPU: hassaku_b200.train.trainer.Trainer')
        if not isinstance(model, SGDMatrixFactorization):
            raise TypeError('ShardedTrainer drives hassaku_b200 SGDMatrixFactorization models only')
        kind = getattr(rec_loss, 'loss_kind', None)
        if kind not in _C.LOSS_KINDS:
            raise ValueError(f'{type(rec_loss).__name__} has no fused kernel (loss kinds: {sorted(_C.LOSS_KINDS)})')
        if conf['optimizer'] not in ('adamw', 'adam'):
            raise ValueError(f"Optimizer {conf['optimizer']} is not available in the sharded step (adamw / adam)")
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.device = torch.device('cuda', torch.cuda.current_device())
        self.rec_loss, self.loss_kind = rec_loss, kind
        self.lr, self.wd = conf['lr'], conf['wd']
        self.decoupled = conf['optimizer'] == 'adamw'
        self.n_epochs = conf['n_epochs']
        self.optimizing_metric = conf['optimizing_metric']
        self.max_patience = conf['max_patience']
        self.model_path = conf['model_path']
        self.exchange = conf.get('sharded_exchange', 'auto')
        if self.exchange not in self.EXCHANGES:
            raise ValueError(f'sharded_exchange {self.exchange!r} not in {self.EXCHANGES}')
        self.eval_precision = conf.get('eval_precision', 'fp32')
        self.pointer_to_model = model          # the full model object: receives the best weights at the end of fit()

        # ---- tables: every rank keeps its rows of the (identically initialised) full model ----
        flags = (model.use_user_bias, model.use_item_bias, model.use_global_bias)
        self.smf = ShardedMF(model.n_users, model.n_items, model.embedding_dim, *flags, world=self.world, rank=self.rank,
                             device=self.device, group=group)
        self.smf.load_full_state_dict({k: v.detach() for k, v in model.state_dict().items()})

        # ---- data: the interactions of this rank's users, local user rows, global item ids ----
        full = train_loader.dataset
        sampler = train_loader.interaction_sampler
        G, r = self.world, self.rank
        local_csr = sp.csr_matrix(sp.csr_matrix(full.sampling_matrix)[np.arange(r, full.n_users, G)])
        sub = TrainRecDataset.from_interactions(local_csr)
        sub.pop_distribution = full.pop_distribution          # popularity sampling stays global
        self.global_batch = int(train_loader.batch_size)
        self.local_batch = max(1, self.global_batch // G)
        local_sampler = NegativeSampler(sub, sampler.n_neg, sampler.neg_sampling_strategy, sampler.squashing_factor_pop_sampling,
                                        getattr(sampler, 'distinct_in_row', True))
        self.loader = TrainDataLoader(local_sampler, sub, batch_size=self.local_batch, shuffle=True, drop_last=True,
                                      device=self.device, seed=int(conf.get('seed', 64)) * 1009 + r)
        n = torch.tensor([len(self.loader)], dtype=torch.int64, device=self.device)
        dist.all_reduce(n, op=dist.ReduceOp.MIN, group=group)
        self.steps_per_epoch = int(n.item())
        if self.steps_per_epoch < 1:
            raise ValueError(f'train_batch_size {self.global_batch} / {G} ranks exceeds the interactions of a rank')
        self.neg_shift = float(rec_loss.neg_shift()) if hasattr(rec_loss, 'neg_shift') else 0.0
        self.val_dataset = val_loader.dataset
        self.eval_batch = int(getattr(val_loader, 'batch_size', 8192))
        self.best_value = self.best_metrics = self.best_epoch = None
        # 'auto' takes the peer exchange only if every rank can map its peers' memory (collective check, once)
        self._peer_ok = self.smf.peer_supported()
        if self._peer_ok and self.exchange == 'auto':
            try:
                self.smf._peer_setup()
            except _C.HskError as ex:
                self._peer_ok = False
                if self.rank == 0:
                    logging.warning(f'peer exchange unavailable, using the all-to-all exchange: {ex}')
        if self.rank == 0:
            logging.info(f'Built ShardedTrainer: world={G}, global batch={self.local_batch * G} ({self.local_batch} per rank), '
                         f'steps per epoch={self.steps_per_epoch}, exchange={self._exchange_name()}')

    # ---- helpers ----
    def _exchange_name(self) -> str:
        ex = self.exchange
        if ex == 'auto':
            n_slots = self.local_batch * (self.loader.interaction_sampler.n_neg + 1)
            if n_slots >= 2 * self.smf.spec.n_items // self.world:
                ex = 'dense'               # the batch covers the item table (ShardedMF.step's rule)
            else:
                ex = 'peer' if self._peer_ok else 'sparse'
        return ex + '_graph'

    def _train_one_epoch(self) -> dict:
        G, r = self.world, self.rank
        ex = self._exchange_name()
        B_global = self.local_batch * G
        it = iter(self.loader)
        for _ in range(self.steps_per_epoch):
            u_local, i_idxs, _labels = next(it)
            self.smf.step(u_local * G + r, i_idxs, B_global, self.loss_kind, self.neg_shift, self.lr, self.wd,
                          decoupled=self.decoupled, exchange=ex)
        rec = self.smf.pop_loss() / self.steps_per_epoch          # the only host sync of the epoch (one all-reduce)
        self.smf.check_status()
        self.loader.check_status()
        return {'epoch_train_loss': rec, 'epoch_train_rec_loss': rec, 'epoch_train_reg_loss': 0.0}

    @torch.no_grad()
    def val(self) -> dict:
        ds = self.val_dataset
        evaluator = FullEvaluator(aggr_by_group=True, n_groups=ds.n_user_groups, user_to_user_group=ds.user_to_user_group)
        lay = self.smf.layout
        replica_bytes = self.smf.spec.n_items * lay.ld * 4 * 2
        free = torch.cuda.mem_get_info(self.device)[0]
        if replica_bytes < free // 4:
            return self.smf.evaluate_replicated(ds.iteration_matrix, ds.exclude_data, evaluator, batch_size=max(self.eval_batch, 1024),
                                                precision=self.eval_precision)
        return self.smf.evaluate(ds.iteration_matrix, ds.exclude_data, evaluator, batch_size=max(self.eval_batch, 1024),
                                 precision=self.eval_precision)

    def _save(self):
        sd = self.smf.full_state_dict(to_cpu=True)      # collective: every rank calls it
        if self.rank == 0:
            os.makedirs(self.model_path, exist_ok=True)
            torch.save(sd, os.path.join(self.model_path, MODEL_FILE))
            print('Model Saved')
        return sd

    def fit(self) -> dict:
        """train/trainer.py:85-185: validation before any update (epoch -1), then up to n_epochs epochs with early stopping
        on `optimizing_metric` and a checkpoint of every new best model.  Returns `best_metrics` on every rank."""
        say = print if self.rank == 0 else (lambda *a, **k: None)
        first = self.val()
        self.best_value = first['max_optimizing_metric'] = first[self.optimizing_metric]
        self.best_epoch = first['best_epoch'] = -1
        self.best_metrics = first
        say('Init - Avg Val Value {:.3f} \n'.format(self.best_value))
        best_sd = self._save()
        patience = self.max_patience
        for epoch in range(self.n_epochs):
            if patience == 0:
                say('Ran out of patience, Stopping ')
                break
            losses = self._train_one_epoch()
            say('Epoch {} - Epoch Avg Train Loss {:.4f} ({:.4f} Rec Loss + {:.4f} Reg Loss )\n'.format(
                epoch, losses['epoch_train_loss'], losses['epoch_train_rec_loss'], losses['epoch_train_reg_loss']))
            metrics = self.val()
            value = metrics[self.optimizing_metric]
            say('Epoch {} - Avg Val Value {:.4f} \n'.format(epoch, value))
            if value > self.best_value:
                self.best_value, self.best_epoch, self.best_metrics = value, epoch, metrics
                metrics['max_optimizing_metric'], metrics['best_epoch'] = value, epoch
                say('Epoch {} - New best model found (val value {:.4f}) \n'.format(epoch, value))
                best_sd = self._save()
                patience = self.max_patience
            else:
                metrics['max_optimizing_metric'] = self.best_value
                patience -= 1
        # like the reference after fit(): the model object holds... the LAST weights there; here the caller's full model gets
        # the BEST ones (what run_train_val reloads from model.pth right after, experiment_helper.py)
        self.pointer_to_model.load_state_dict(best_sd)
        return self.best_metrics

    def close(self):
        self.smf.close()
