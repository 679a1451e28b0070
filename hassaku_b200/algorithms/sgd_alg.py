"""SGDMatrixFactorization behind the reference API (algorithms/sgd_alg.py:110-184), computed by the sm_100a kernels.

Storage (B200-first): every parameter of the model lives in ONE flat fp32 arena

    [ Uw (n_users x ld) | Vw (n_items x ld) | Ub (n_users) | Ib (n_items) | Gb (1) ]      ld = ceil4(embedding_dim)

so that (a) rows are 16-byte aligned for 128-bit gathers / vector reductions even for d = 402, (b) the optimizer is a
single streaming pass over one contiguous range, (c) m, v and the dense gradient are arenas of the same layout.
`user_embeddings.weight` etc. are `[rows, d]` strided views of the arena, so `state_dict()` / `model.pth` keep the
reference's names and shapes (base_classes.py:156-165).  Pad columns are zero and stay zero.
"""
import logging
from typing import Tuple, Union

import torch
from torch import nn

from hassaku_b200 import _C, determinism
from hassaku_b200.algorithms.base_classes import SGDBasedRecommenderAlgorithm
from hassaku_b200.train.utils import general_weight_init


def _align_up(x: int, a: int) -> int:
    return (x + a - 1) // a * a


class ArenaLayout:
    """Element offsets of the tables inside the flat arena (segments 128-byte aligned)."""
    ALIGN = 32

    def __init__(self, n_users: int, n_items: int, d: int, use_user_bias: bool, use_item_bias: bool,
                 use_global_bias: bool):
        self.n_users, self.n_items, self.d = n_users, n_items, d
        self.ld = _align_up(d, 4)
        off = 0
        self.off_U = off
        off = _align_up(off + n_users * self.ld, self.ALIGN)
        self.off_V = off
        off = _align_up(off + n_items * self.ld, self.ALIGN)
        self.off_Ub = self.off_Ib = self.off_Gb = -1
        if use_user_bias:
            self.off_Ub = off
            off = _align_up(off + n_users, self.ALIGN)
        if use_item_bias:
            self.off_Ib = off
            off = _align_up(off + n_items, self.ALIGN)
        if use_global_bias:
            self.off_Gb = off
            off = _align_up(off + 1, self.ALIGN)
        self.n_total = off

    def views(self, arena: torch.Tensor):
        """(Uw [U, d] strided, Vw [I, d] strided, Ub [U, 1] | None, Ib [I, 1] | None, Gb [1] | None)."""
        U, I, d, ld = self.n_users, self.n_items, self.d, self.ld
        Uw = arena[self.off_U:self.off_U + U * ld].view(U, ld)[:, :d]
        Vw = arena[self.off_V:self.off_V + I * ld].view(I, ld)[:, :d]
        Ub = arena[self.off_Ub:self.off_Ub + U].view(U, 1) if self.off_Ub >= 0 else None
        Ib = arena[self.off_Ib:self.off_Ib + I].view(I, 1) if self.off_Ib >= 0 else None
        Gb = arena[self.off_Gb:self.off_Gb + 1] if self.off_Gb >= 0 else None
        return Uw, Vw, Ub, Ib, Gb

    def tables(self, arena: torch.Tensor) -> _C.MfTables:
        Uw, Vw, Ub, Ib, Gb = self.views(arena)
        return _C.make_tables(Uw, Vw, Ub, Ib, Gb, self.d)


class _MfScoreFn(torch.autograd.Function):
    """forward = hsk_mf_scores; backward = hsk_mf_scatter_grads into fresh dense gradient tables (what autograd +
    aten::embedding_dense_backward do in the reference, SURVEY §2b K4); hsk_mf_scatter_grads_det under
    torch.use_deterministic_algorithms(True)."""

    @staticmethod
    def forward(ctx, model, u_idxs, i_idxs, Uw, Vw, Ub, Ib, Gb):
        scores = torch.empty(i_idxs.shape, dtype=torch.float32, device=i_idxs.device)
        _C.mf_scores(model._tables(), u_idxs, i_idxs, scores, model._status())
        ctx.model = model
        ctx.save_for_backward(u_idxs, i_idxs)
        return scores

    @staticmethod
    def backward(ctx, dscores):
        model = ctx.model
        u_idxs, i_idxs = ctx.saved_tensors
        lay = model.layout
        g_arena = torch.zeros(lay.n_total, dtype=torch.float32, device=dscores.device)
        if determinism.enabled():
            scratch = determinism.scratch(model, _C.det_scratch_bytes(i_idxs.shape[0], i_idxs.shape[1], lay.ld),
                                          dscores.device)
            _C.mf_scatter_grads_det(model._tables(), lay.tables(g_arena), u_idxs, i_idxs, dscores.contiguous().float(),
                                    scratch, model._status())
        else:
            _C.mf_scatter_grads(model._tables(), lay.tables(g_arena), u_idxs, i_idxs,
                                dscores.contiguous().float(), model._status())
        grads = lay.views(g_arena)   # (gU, gV, gUb, gIb, gGb); None where the model has no such table
        need = ctx.needs_input_grad[3:]
        return (None, None, None) + tuple(g if n else None for g, n in zip(grads, need))


class SGDMatrixFactorization(SGDBasedRecommenderAlgorithm):
    """Matrix factorization trained with SGD — same constructor, parameter names, methods and initialisation as
    the reference (algorithms/sgd_alg.py:110-184); `forward` runs the fused gather-score kernel."""

    def __init__(self, n_users: int, n_items: int, embedding_dim: int = 100, use_user_bias: bool = False,
                 use_item_bias: bool = False, use_global_bias: bool = False, *, _device=None, _seed: int = 64,
                 _std=None):
        super().__init__()
        self.n_users = n_users
        self.n_items = n_items
        self.embedding_dim = embedding_dim
        self.use_user_bias = use_user_bias
        self.use_item_bias = use_item_bias
        self.use_global_bias = use_global_bias
        if embedding_dim > 1024:
            raise ValueError('hassaku_b200 supports embedding_dim <= 1024')

        self.layout = ArenaLayout(n_users, n_items, embedding_dim, use_user_bias, use_item_bias, use_global_bias)
        if _device is not None:
            # large tables (cfg4: 385 M, cfg5: 2.8 G parameters): no host copy — the modules are created without storage
            # and the arena is drawn directly on the device with the reference's distribution N(0, (0.1 / shape[-1])^2)
            # (train/utils.py:11-13).  Same distribution, NOT the same bits as the host constructor (different generator).
            with torch.device('meta'):
                self.user_embeddings = nn.Embedding(self.n_users, self.embedding_dim)
                self.item_embeddings = nn.Embedding(self.n_items, self.embedding_dim)
                if self.use_user_bias:
                    self.user_bias = nn.Embedding(self.n_users, 1)
                if self.use_item_bias:
                    self.item_bias = nn.Embedding(self.n_items, 1)
                if self.use_global_bias:
                    self.global_bias = nn.Parameter(torch.zeros(1), requires_grad=True)
            arena = torch.zeros(self.layout.n_total, dtype=torch.float32, device=_device)
            gen = torch.Generator(device=arena.device)
            gen.manual_seed(int(_seed))
            for j, view in enumerate(self.layout.views(arena)[:4]):     # Uw, Vw, Ub, Ib
                if view is not None:
                    std = 0.1 / view.shape[-1] if _std is None else _std[0 if j < 2 else 1]
                    view.normal_(0., std, generator=gen)
        else:
            # Same module construction + init order as the reference (sgd_alg.py:127-138, train/utils.py:11-13), so the
            # same torch seed yields bit-identical initial weights.
            self.user_embeddings = nn.Embedding(self.n_users, self.embedding_dim)
            self.item_embeddings = nn.Embedding(self.n_items, self.embedding_dim)
            if self.use_user_bias:
                self.user_bias = nn.Embedding(self.n_users, 1)
            if self.use_item_bias:
                self.item_bias = nn.Embedding(self.n_items, 1)
            self.apply(general_weight_init)
            if self.use_global_bias:
                self.global_bias = nn.Parameter(torch.zeros(1), requires_grad=True)
            arena = torch.zeros(self.layout.n_total, dtype=torch.float32)
            Uw, Vw, Ub, Ib, Gb = self.layout.views(arena)
            with torch.no_grad():
                Uw.copy_(self.user_embeddings.weight)
                Vw.copy_(self.item_embeddings.weight)
                if Ub is not None:
                    Ub.copy_(self.user_bias.weight)
                if Ib is not None:
                    Ib.copy_(self.item_bias.weight)
        self._status_flag = None
        self._set_arena(arena)

        self.name = 'SGDMatrixFactorization'
        logging.info(f'Built {self.name} module\n'
                     f'- embedding_dim: {self.embedding_dim} \n'
                     f'- use_user_bias: {self.use_user_bias} \n'
                     f'- use_item_bias: {self.use_item_bias} \n'
                     f'- use_global_bias: {self.use_global_bias}')

    @classmethod
    def on_device(cls, n_users: int, n_items: int, embedding_dim: int, use_user_bias: bool = False,
                  use_item_bias: bool = False, use_global_bias: bool = False, device='cuda', seed: int = 64, std=None):
        """The model with its arena allocated and initialised ON `device` (for tables too large to build on the host).
        `std` = (embedding std, bias std) overrides the reference's 0.1 / shape[-1] (evaluation benchmarks use
        (1 / sqrt(d), 0.05): with the training init every user's ranking would be the item-bias ranking)."""
        return cls(n_users, n_items, embedding_dim, use_user_bias, use_item_bias, use_global_bias, _device=device, _seed=seed,
                   _std=std)

    # ---- arena plumbing ----
    def _set_arena(self, arena: torch.Tensor):
        self._arena = arena
        Uw, Vw, Ub, Ib, Gb = self.layout.views(arena)
        self.user_embeddings.weight = nn.Parameter(Uw)
        self.item_embeddings.weight = nn.Parameter(Vw)
        if Ub is not None:
            self.user_bias.weight = nn.Parameter(Ub)
        if Ib is not None:
            self.item_bias.weight = nn.Parameter(Ib)
        if Gb is not None:
            self.global_bias = nn.Parameter(Gb)
        self._tables_cache = None
        self._status_flag = None

    def _apply(self, fn, recurse=True):
        # .to() / .cuda() / .float(): move the arena as a whole and re-create the parameter views (the default
        # implementation would move every parameter separately and break the single-arena layout)
        self._set_arena(fn(self._arena.detach()))
        return self

    @property
    def arena(self) -> torch.Tensor:
        return self._arena

    def _tables(self) -> _C.MfTables:
        if self._tables_cache is None:
            self._tables_cache = self.layout.tables(self._arena)
        return self._tables_cache

    def _status(self) -> torch.Tensor:
        if self._status_flag is None or self._status_flag.device != self._arena.device:
            self._status_flag = torch.zeros(1, dtype=torch.int32, device=self._arena.device)
        return self._status_flag

    def check_status(self):
        """Host sync: raises IndexError if any kernel met an out-of-range index since the last check (the reference
        raises from torch at the embedding lookup)."""
        if self._status_flag is not None:
            st = int(self._status_flag.item())
            if st & _C.STATUS_BAD_INDEX:
                self._status_flag.zero_()
                raise IndexError('index out of range in SGDMatrixFactorization (user or item index)')

    def state_dict(self, *args, **kwargs):
        sd = super().state_dict(*args, **kwargs)
        for k, v in list(sd.items()):
            if isinstance(v, torch.Tensor) and not v.is_contiguous():
                sd[k] = v.detach().contiguous()  # do not serialise the whole arena once per view
        return sd

    # ---- reference API ----
    def get_user_representations(self, u_idxs: torch.Tensor) -> Union[torch.Tensor, Tuple[torch.Tensor, ...]]:
        # sgd_alg.py:148-152 (materialising accessor kept for API compatibility; `forward` never calls it)
        if self.use_user_bias:
            return self.user_embeddings(u_idxs), self.user_bias(u_idxs)
        return self.user_embeddings(u_idxs)

    def get_item_representations(self, i_idxs: torch.Tensor) -> Union[torch.Tensor, Tuple[torch.Tensor, ...]]:
        # sgd_alg.py:154-157
        if self.use_item_bias:
            return self.item_embeddings(i_idxs), self.item_bias(i_idxs).squeeze()
        return self.item_embeddings(i_idxs)

    def combine_user_item_representations(self, u_repr, i_repr) -> torch.Tensor:
        # sgd_alg.py:159-179
        u_embed, u_bias = u_repr if isinstance(u_repr, tuple) else (u_repr, None)
        i_embed, i_bias = i_repr if isinstance(i_repr, tuple) else (i_repr, None)
        out = (u_embed[:, None, :] * i_embed).sum(dim=-1)
        if self.use_user_bias:
            out += u_bias
        if self.use_item_bias:
            out += i_bias
        if self.use_global_bias:
            out += self.global_bias
        return out

    def forward(self, u_idxs: torch.Tensor, i_idxs: torch.Tensor) -> torch.Tensor:
        """base_classes.py:99-108 — u_idxs int64 [B], i_idxs int64 [B, 1+N] -> fp32 [B, 1+N], differentiable.
        One fused gather-score kernel (hsk_mf_scores); no [B, N+1, d] intermediate."""
        if not self._arena.is_cuda:
            raise _C.HskError('SGDMatrixFactorization.forward needs the model on a CUDA device '
                              '(hassaku_b200 has no CPU path): call model.to("cuda")')
        squeeze = i_idxs.dim() == 1
        if squeeze:
            i_idxs = i_idxs.unsqueeze(1)
        u_idxs = u_idxs.to(self._arena.device, torch.int64).contiguous()
        i_idxs = i_idxs.to(self._arena.device, torch.int64).contiguous()
        Ub = self.user_bias.weight if self.use_user_bias else None
        Ib = self.item_bias.weight if self.use_item_bias else None
        Gb = self.global_bias if self.use_global_bias else None
        out = _MfScoreFn.apply(self, u_idxs, i_idxs, self.user_embeddings.weight, self.item_embeddings.weight, Ub, Ib,
                               Gb)
        return out.squeeze(1) if squeeze else out

    @staticmethod
    def build_from_conf(conf: dict, dataset):
        # sgd_alg.py:181-184
        return SGDMatrixFactorization(dataset.n_users, dataset.n_items, conf['embedding_dim'], conf['use_user_bias'],
                                      conf['use_item_bias'], conf['use_global_bias'])


class SGDBaseline(SGDMatrixFactorization):
    """Bias-only baseline `user_bias[u] + item_bias[i] + global_bias` (algorithms/sgd_alg.py:72-107) on the SAME kernels:
    it is the matrix factorization with embedding_dim 1 whose two embedding tables are identically zero.  Zero
    embeddings stay exactly zero under every supported optimizer (their gradient ds * 0 is 0, so m = v = 0 and the
    Adam / Adagrad update 0 / (0 + eps) is 0; weight decay of 0 is 0), so training, the fused step, the sharded step and
    the full-rank evaluator all work unchanged.  Parameters, `state_dict()` names / shapes and the initialisation order
    are the reference's (`user_bias.weight [U, 1]`, `item_bias.weight [I, 1]`, `global_bias [1]`); the zero tables are
    plain tensors inside the arena, not parameters."""

    def __init__(self, n_users: int, n_items: int):
        SGDBasedRecommenderAlgorithm.__init__(self)
        self.n_users = n_users
        self.n_items = n_items
        self.embedding_dim = 1
        self.use_user_bias = self.use_item_bias = self.use_global_bias = True
        # reference construction order (sgd_alg.py:83-87): same torch seed -> bit-identical initial weights
        self.user_bias = nn.Embedding(self.n_users, 1)
        self.item_bias = nn.Embedding(self.n_items, 1)
        self.global_bias = nn.Parameter(torch.zeros(1), requires_grad=True)
        self.apply(general_weight_init)

        self.layout = ArenaLayout(n_users, n_items, 1, True, True, True)
        arena = torch.zeros(self.layout.n_total, dtype=torch.float32)
        _, _, Ub, Ib, Gb = self.layout.views(arena)
        with torch.no_grad():
            Ub.copy_(self.user_bias.weight)
            Ib.copy_(self.item_bias.weight)
            Gb.copy_(self.global_bias)
        self._status_flag = None
        self._set_arena(arena)
        self.name = 'SGDBaseline'
        logging.info(f'Built {self.name} module\n')

    def _set_arena(self, arena: torch.Tensor):
        self._arena = arena
        Uw, Vw, Ub, Ib, Gb = self.layout.views(arena)
        # the zero embedding tables: attributes with a `.weight`, like nn.Embedding, for the code that reads
        # `alg.user_embeddings.weight` (TopKScorer); not registered as modules / parameters
        object.__setattr__(self, 'user_embeddings', _FrozenTable(Uw))
        object.__setattr__(self, 'item_embeddings', _FrozenTable(Vw))
        self.user_bias.weight = nn.Parameter(Ub)
        self.item_bias.weight = nn.Parameter(Ib)
        self.global_bias = nn.Parameter(Gb)
        self._tables_cache = None
        self._status_flag = None

    def get_user_representations(self, u_idxs: torch.Tensor) -> torch.Tensor:
        return self.user_bias(u_idxs)                       # sgd_alg.py:93-94

    def get_item_representations(self, i_idxs: torch.Tensor) -> torch.Tensor:
        return self.item_bias(i_idxs).squeeze()             # sgd_alg.py:96-97

    def combine_user_item_representations(self, u_repr, i_repr) -> torch.Tensor:
        return u_repr + i_repr + self.global_bias           # sgd_alg.py:99-102

    def forward(self, u_idxs: torch.Tensor, i_idxs: torch.Tensor) -> torch.Tensor:
        if not self._arena.is_cuda:
            raise _C.HskError('SGDBaseline.forward needs the model on a CUDA device (hassaku_b200 has no CPU path): '
                              'call model.to("cuda")')
        squeeze = i_idxs.dim() == 1
        if squeeze:
            i_idxs = i_idxs.unsqueeze(1)
        u_idxs = u_idxs.to(self._arena.device, torch.int64).contiguous()
        i_idxs = i_idxs.to(self._arena.device, torch.int64).contiguous()
        out = _MfScoreFn.apply(self, u_idxs, i_idxs, None, None, self.user_bias.weight, self.item_bias.weight,
                               self.global_bias)
        return out.squeeze(1) if squeeze else out

    @staticmethod
    def build_from_conf(conf: dict, dataset):
        return SGDBaseline(dataset.n_users, dataset.n_items)   # sgd_alg.py:104-106


class _FrozenTable:
    """`.weight` holder for the all-zero embedding tables of SGDBaseline (a view of the arena, never trained)."""

    def __init__(self, weight: torch.Tensor):
        self.weight = weight
