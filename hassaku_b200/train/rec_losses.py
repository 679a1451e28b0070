"""Recommendation losses behind the reference API (train/rec_losses.py:12-145), computed by hsk_rec_loss.

`compute_loss(logits, labels)` returns a 0-dim tensor with autograd (one kernel produces the loss and dL/dlogits);
dtype follows the reference: float64 for bpr/bce when the loader's float64 labels are passed (SURVEY A.2), float32 for
sampled-softmax."""
import logging
import math
from abc import ABC, abstractmethod
from enum import Enum

import torch

from hassaku_b200 import _C, determinism


class RecommenderSystemLoss(ABC):
    """Interface of the reference's loss objects (rec_losses.py:12-25): `compute_loss(logits, labels)` and the
    `build_from_conf(conf, dataset)` factory; `.name` is the class name.  `loss_kind` / `neg_shift()` are what the fused
    Trainer path hands to hsk_mf_train_fused instead of calling `compute_loss`."""
    loss_kind = None

    def __init__(self):
        self.name = type(self).__name__
        logging.info('Built %s module', self.name)

    def neg_shift(self) -> float:
        return 0.0

    @abstractmethod
    def compute_loss(self, logits: torch.Tensor, labels: torch.Tensor):
        """logits fp32 [B, 1 + N] (column 0 = positive), labels [B, 1 + N] -> 0-dim loss tensor with autograd."""

    @staticmethod
    @abstractmethod
    def build_from_conf(conf: dict, dataset):
        """Factory used by `RecommenderSystemLossesEnum[...].value.build_from_conf` (experiment_helper.py:42)."""


def _promoted(logits: torch.Tensor, labels) -> torch.dtype:
    # the reference's BCEWithLogits on float64 labels returns float64 (SURVEY A.2)
    return torch.promote_types(logits.dtype, labels.dtype) if labels is not None else logits.dtype


class _RecLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, kind, shift, out_dtype, mutate):
        if not logits.is_cuda:
            raise _C.HskError('hassaku_b200 losses need CUDA tensors (no CPU path)')
        x = logits.detach()
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
            mutate = False
        lab = None
        if labels is not None and kind != _C.LOSS_KINDS['sampled_softmax']:
            lab = labels.detach().to(x.device, torch.float64).contiguous()
        loss = torch.zeros(1, dtype=torch.float64, device=x.device)
        ds = torch.empty_like(x)
        if determinism.enabled():   # fixed-order sum of the per-row losses
            scratch = torch.empty(8 * x.shape[0], dtype=torch.uint8, device=x.device)
            _C.rec_loss_det(x, lab, kind, shift, 1.0, loss, ds, scratch, x if mutate else None)
        else:
            _C.rec_loss(x, lab, kind, shift, 1.0, loss, ds, x if mutate else None)
        # (the in-place shift goes through the detached alias: nothing upstream saved the model output)
        ctx.save_for_backward(ds)
        return loss[0].to(out_dtype)

    @staticmethod
    def backward(ctx, grad_out):
        (ds,) = ctx.saved_tensors
        return ds * grad_out.to(torch.float32), None, None, None, None, None


def _apply(logits, labels, kind, shift, out_dtype, mutate=False):
    return _RecLossFn.apply(logits, labels, kind, shift, out_dtype, mutate)


class RecBinaryCrossEntropy(RecommenderSystemLoss):
    """rec_losses.py:28-53: BCEWithLogits over all B*(1+N) logits."""
    loss_kind = 'bce'

    def compute_loss(self, logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        return _apply(logits, labels, _C.LOSS_KINDS[self.loss_kind], 0.0, _promoted(logits, labels))

    @staticmethod
    def build_from_conf(conf: dict, dataset):
        return RecBinaryCrossEntropy()


class RecBayesianPersonalizedRankingLoss(RecommenderSystemLoss):
    """rec_losses.py:56-88: mean over B*N of -log sigmoid(pos - neg)."""
    loss_kind = 'bpr'

    def compute_loss(self, logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        return _apply(logits, labels, _C.LOSS_KINDS[self.loss_kind], 0.0, _promoted(logits, labels))

    @staticmethod
    def build_from_conf(conf: dict, dataset):
        return RecBayesianPersonalizedRankingLoss()


class RecSampledSoftmaxLoss(RecommenderSystemLoss):
    """rec_losses.py:91-139: -x_pos + logsumexp(x + [neg] * ln(n_items / neg_train)), mean over B.  Like the
    reference (:134) the shift is applied to `logits[:, 1:]` IN PLACE (SURVEY Appendix C.7)."""
    loss_kind = 'sampled_softmax'

    def __init__(self, n_items: int = None, train_neg_strategy: str = None, neg_train: int = None):
        super().__init__()
        self.n_items, self.train_neg_strategy, self.neg_train = n_items, train_neg_strategy, neg_train

    @staticmethod
    def build_from_conf(conf: dict, dataset):
        return RecSampledSoftmaxLoss(n_items=dataset.n_items, train_neg_strategy=conf['train_neg_strategy'],
                                     neg_train=conf['neg_train'])

    def neg_shift(self) -> float:
        if self.train_neg_strategy == 'uniform':
            return math.log(self.n_items / self.neg_train)
        return 0.0

    def compute_loss(self, logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        shift = self.neg_shift()
        return _apply(logits, None, _C.LOSS_KINDS['sampled_softmax'], shift, torch.float32, mutate=shift != 0.0)


class RecommenderSystemLossesEnum(Enum):
    bce = RecBinaryCrossEntropy
    bpr = RecBayesianPersonalizedRankingLoss
    sampled_softmax = RecSampledSoftmaxLoss
