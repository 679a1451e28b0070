"""Dense Adam / AdamW over the model's flat parameter arena — torch.optim.AdamW / torch.optim.Adam semantics
(train/trainer.py:48-53) in ONE streaming kernel (hsk_adamw_dense / hsk_adamw_dense_rows): every element is updated
every step, zero-gradient rows included (SURVEY A.5), and the gradient arena is zeroed in the same pass (replaces
optimizer.zero_grad()).  When a batch touches a small part of a table (cfg4: 0.35 M of 3 M rows) the rows kernel skips
the gradient READ and re-zeroing of the untouched rows — their gradient is exactly zero, so the result is bit-identical
to the plain dense kernel at 24 instead of 32 bytes per parameter.  With `state_lag` K > 1 (AdamW, or Adam without
weight decay) those rows also write m and v back only once every K steps (hsk_adamw_dense_rows_lag): 16 + 8 / K bytes per
parameter.  p is current after every step, and `m` / `v` bring every row up to date before they are returned."""
import torch

from hassaku_b200 import _C

# m / v write-back period of untouched rows (DenseAdam state_lag), measured at cfg4: profiles/adamw_lag_cost.json
DEFAULT_STATE_LAG = 8


def stamp_segments(lay, B: int, n_slots: int, stamp_users, stamp_items):
    """(segments, stamps_users | None, stamps_items | None) for a batch of B samples and n_slots item slots: the row
    segments of arena layout `lay` whose untouched rows skip the gradient traffic — only a table the batch covers
    sparsely (otherwise the plain streaming pass is at least as fast and no marking launch is spent)."""
    su = stamp_users if 4 * B <= lay.n_users else None
    si = stamp_items if n_slots <= lay.n_items else None
    segs = []
    if su is not None:
        segs.append((lay.off_U, lay.n_users, lay.ld, su))
    if si is not None:
        segs.append((lay.off_V, lay.n_items, lay.ld, si))
    return tuple(segs), su, si


class DenseAdam(torch.optim.Optimizer):
    """`decoupled=True` -> torch.optim.AdamW(lr, weight_decay); False -> torch.optim.Adam(lr, weight_decay) (L2).
    Defaults as torch: betas (0.9, 0.999), eps 1e-8, AdamW weight_decay default is whatever the caller passes
    (the reference always passes conf['wd'])."""

    def __init__(self, model, lr: float = 1e-3, weight_decay: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8,
                 decoupled: bool = True, arith: int = 0, mode: str = 'dense', state_lag: int = DEFAULT_STATE_LAG):
        if not 1 <= int(state_lag) <= 128:
            raise ValueError('state_lag must be in [1, 128]')
        self.model = model
        super().__init__(list(model.parameters()),
                         dict(lr=lr, weight_decay=weight_decay, betas=betas, eps=eps, decoupled=decoupled))
        self.arith = arith
        if mode not in ('dense', 'lazy'):
            raise ValueError("optimizer_mode must be 'dense' (torch-faithful) or 'lazy' (row-sparse)")
        if mode == 'lazy' and not decoupled:
            raise ValueError('lazy mode is defined for AdamW (decoupled decay) only')
        self.mode = mode
        self.state_lag = int(state_lag) if mode == 'dense' else 1
        self._t = 0
        self._segments = ()      # row segments whose untouched rows skip the gradient traffic in the NEXT step_fused
        self._behind = {}        # segment offset -> segment: tables whose rows' m / v may be older than step t
        self._lag_key = None     # (beta1, beta2, arith, lag) the rows of _behind were stepped with
        self._base_t = {}        # segment offset -> the step that base_in holds for every row of the table
        self._alloc()

    def _alloc(self):
        arena = self.model.arena
        if not arena.is_cuda:
            raise _C.HskError('DenseAdam needs the model on a CUDA device (no CPU path)')
        self._m = torch.zeros_like(arena)
        self._v = torch.zeros_like(arena)
        self.g = torch.zeros_like(arena)
        self.grad_tables = self.model.layout.tables(self.g)
        lay = self.model.layout
        if self.mode == 'lazy':
            self.touched_users = torch.zeros(lay.n_users, dtype=torch.uint8, device=arena.device)
            self.touched_items = torch.zeros(lay.n_items, dtype=torch.uint8, device=arena.device)
        else:   # per-row step stamps (hsk_row_stamp): never cleared
            self.stamp_users = torch.zeros(lay.n_users, dtype=torch.uint8, device=arena.device)
            self.stamp_items = torch.zeros(lay.n_items, dtype=torch.uint8, device=arena.device)
            if self.state_lag > 1:   # per row the step & 255 of its last m / v write-back: [base_in, base_out]
                self._bases = {off: [torch.zeros(rows, dtype=torch.uint8, device=arena.device) for _ in range(2)]
                               for off, rows in ((lay.off_U, lay.n_users), (lay.off_V, lay.n_items))}

    @property
    def t(self):
        return self._t

    @t.setter
    def t(self, step: int):
        self.sync_state()
        self._t = int(step)

    @property
    def m(self):
        """first moments of the arena, every row current"""
        self.sync_state()
        return self._m

    @property
    def v(self):
        """second moments of the arena, every row current"""
        self.sync_state()
        return self._v

    def sync_state(self):
        """Bring the m and v of every row to step t (rows the last steps did not write back are behind)."""
        if not self._behind:
            return
        segs = tuple(self._behind.values())
        b1, b2, arith, _ = self._lag_key
        _C.adamw_lag_sync(self._m, self._v, segs, [self._bases[sg[0]] for sg in segs], b1, b2, self._t, arith=arith)
        for sg in segs:
            self._swap_bases(sg[0])
        self._behind = {}

    def _swap_bases(self, off):
        b = self._bases[off]
        b[0], b[1] = b[1], b[0]
        self._base_t[off] = self._t

    @property
    def grad_views(self):
        """(gU, gV, gUb, gIb, gGb) views of the dense gradient arena, shaped like the parameters."""
        return self.model.layout.views(self.g)

    def mark(self, u_idxs: torch.Tensor, i_idxs: torch.Tensor):
        """Remember which rows this batch's gradients touch (call between the scatter and step_fused).
        lazy mode: the rows to update.  dense mode: the rows whose gradient must be read and re-zeroed — only for a
        table the batch covers sparsely (otherwise the plain streaming pass is at least as fast and no launch is spent)."""
        lay = self.model.layout
        if self.mode == 'lazy':
            _C.mark_touched(u_idxs, i_idxs, lay.n_users, lay.n_items, self.touched_users, self.touched_items)
            return
        segs, su, si = stamp_segments(lay, int(u_idxs.numel()), int(i_idxs.numel()), self.stamp_users, self.stamp_items)
        if segs:
            _C.mark_batch(u_idxs, i_idxs, lay.n_users, lay.n_items, su, si, step=self._t + 1)
        self._segments = segs

    def _step_lazy(self, grp):
        lay, arena = self.model.layout, self.model.arena

        def t2d(a, off, rows):
            return a[off:off + rows * lay.ld].view(rows, lay.ld)

        def vec(a, off, rows):
            return a[off:off + rows] if off >= 0 else None

        for off_t, off_b, rows, touched in ((lay.off_U, lay.off_Ub, lay.n_users, self.touched_users),
                                            (lay.off_V, lay.off_Ib, lay.n_items, self.touched_items)):
            bias = None
            if off_b >= 0:
                bias = tuple(vec(a, off_b, rows) for a in (arena, self._m, self._v, self.g))
            _C.adamw_rows_lazy(t2d(arena, off_t, rows), t2d(self._m, off_t, rows), t2d(self._v, off_t, rows),
                               t2d(self.g, off_t, rows), touched, grp['lr'], grp['betas'][0], grp['betas'][1], grp['eps'],
                               grp['weight_decay'], self._t, bias=bias)
        if lay.off_Gb >= 0:   # the global bias is touched by every sample: plain dense update of that one element
            sl = slice(lay.off_Gb, lay.off_Gb + 4)
            _C.adamw_dense(arena[sl], self._m[sl], self._v[sl], self.g[sl], grp['lr'], grp['betas'][0], grp['betas'][1],
                           grp['eps'], grp['weight_decay'], self._t, arith=self.arith, zero_grad=True)

    def step_fused(self):
        """One optimizer step consuming the gradient arena `self.g` (filled by hsk_mf_train_fused)."""
        grp = self.param_groups[0]
        if self.mode == 'lazy':
            self._t += 1
            return self._step_lazy(grp)
        segs, self._segments = self._segments, ()
        b1, b2 = grp['betas']
        key = (b1, b2, self.arith, self.state_lag)
        lag = self.state_lag > 1 and bool(segs) and (grp['decoupled'] or grp['weight_decay'] == 0.0)
        offs = {sg[0] for sg in segs}
        if self._behind and not (lag and key == self._lag_key and self._behind.keys() <= offs):
            self.sync_state()    # the rows behind are brought up to date with what they were stepped with
        self._t += 1
        p, m, v, g = self.model.arena, self._m, self._v, self.g
        if lag:
            for off in offs:     # a table entering the lagged update: every row's m / v are those of step t - 1
                if self._base_t.get(off) != self._t - 1:
                    self._bases[off][0].fill_((self._t - 1) & 255)
            _C.adamw_dense_rows_lag(p, m, v, g, segs, [self._bases[sg[0]] for sg in segs], self.state_lag, grp['lr'], b1,
                                    b2, grp['eps'], grp['weight_decay'], self._t, arith=self.arith,
                                    adam_l2=not grp['decoupled'])
            for sg in segs:
                self._swap_bases(sg[0])
                self._behind[sg[0]] = sg
            self._lag_key = key
        elif segs:
            _C.adamw_dense_rows(p, m, v, g, segs, grp['lr'], b1, b2, grp['eps'], grp['weight_decay'], self._t,
                                arith=self.arith, adam_l2=not grp['decoupled'])
        else:
            _C.adamw_dense(p, m, v, g, grp['lr'], b1, b2, grp['eps'], grp['weight_decay'], self._t, arith=self.arith,
                           adam_l2=not grp['decoupled'], zero_grad=True)

    @torch.no_grad()
    def step(self, closure=None):
        """torch.optim API: gathers the parameters' `.grad` (autograd path) into the arena, then steps."""
        loss = closure() if closure is not None else None
        lay = self.model.layout
        names = ('user_embeddings.weight', 'item_embeddings.weight', 'user_bias.weight', 'item_bias.weight',
                 'global_bias')
        params = dict(self.model.named_parameters())
        for name, gview in zip(names, lay.views(self.g)):
            if gview is None:
                continue
            p = params[name]
            if p.grad is not None:
                gview.add_(p.grad.view_as(gview))
        self._segments = ()      # autograd gradients are dense: plain streaming pass
        self.step_fused()
        return loss


class DenseAdagrad(torch.optim.Optimizer):
    """torch.optim.Adagrad(lr, weight_decay) (train/trainer.py:50-51) over the flat arena in one streaming kernel."""
    mode = 'dense'

    def __init__(self, model, lr: float = 1e-2, weight_decay: float = 0.0, eps: float = 1e-10):
        self.model = model
        super().__init__(list(model.parameters()), dict(lr=lr, weight_decay=weight_decay, eps=eps))
        arena = model.arena
        if not arena.is_cuda:
            raise _C.HskError('DenseAdagrad needs the model on a CUDA device (no CPU path)')
        self.state_sum = torch.zeros_like(arena)
        self.g = torch.zeros_like(arena)
        self.grad_tables = model.layout.tables(self.g)
        self.t = 0

    def step_fused(self):
        grp = self.param_groups[0]
        self.t += 1
        _C.adagrad_dense(self.model.arena, self.state_sum, self.g, grp['lr'], grp['eps'], grp['weight_decay'], zero_grad=True)

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        names = ('user_embeddings.weight', 'item_embeddings.weight', 'user_bias.weight', 'item_bias.weight', 'global_bias')
        params = dict(self.model.named_parameters())
        for name, gview in zip(names, self.model.layout.views(self.g)):
            if gview is not None and params[name].grad is not None:
                gview.add_(params[name].grad.view_as(gview))
        self.step_fused()
        return loss
