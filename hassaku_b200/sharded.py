"""Item-/user-sharded SGD-MF over the GPUs of one box (SURVEY §8e): one process per GPU, torch.distributed (NCCL over
NVLink / NVSwitch) for the exchanges, the same sm_100a kernels for the arithmetic.  The reference's only multi-GPU
mechanism is nn.DataParallel (train/trainer.py:38-40), which re-broadcasts all parameters every forward and reduces
dense gradients to GPU 0; here nothing is replicated.

Partition (G = world size): item i lives on rank i % G as local row i // G (spreads the Zipf-popular low ids), with its
bias and AdamW state; user u likewise on rank u % G.  A training sample is processed by the owner of its USER, so user
rows, user AdamW state and the negative sampler are always local.

One training step (identical arithmetic to the single-GPU step on the union of the ranks' batches), SPARSE exchange
(cfg4: B (N + 1) << n_items) — every buffer has a fixed shape and nothing syncs with the host, so the step is ONE CUDA
graph (`exchange='sparse_graph'`):
  1. hsk_route_items: distinct item ids of the local batch grouped by owner -> req_rows [G, capq] (-1 padded), and for
     every batch slot its row in the compact table of fetched rows
  2. all-to-all: req_rows -> the owners                                             (int32, G x capq)
  3. owners pack the requested rows + biases (hsk_shard_pack), all-to-all back      (fp32 blocks [G, block_rows, ld])
  4. hsk_mf_train_fused_n on (local user shard, compact table) with GLOBAL normalisers
  5. all-to-all: compact row / bias gradients to the owners, hsk_shard_unpack_add into the local dense gradient
  6. hsk_adamw_dense_rows over the local arena: 24 B / parameter for rows without a gradient, 32 B for the touched ones
     (the dominant term of the step shards perfectly: P / G parameters per GPU)
ORDERED exchange (`exchange='ordered'` / `'ordered_graph'`): the sparse exchange with every floating-point cross-row and
cross-rank reduction in a fixed order — hsk_mf_train_fused_det_n in step 4, hsk_shard_unpack_ordered in step 5, the
global-bias gradient and the loss summed in rank order — so a run gives the same bits every time at a fixed world size
(order contract in include/hassaku_b200.h); the exchange to use under torch.use_deterministic_algorithms(True).
DENSE exchange (cfg2: the batch covers the item table anyway): one all-gather of the [cap + bias rows, ld] blocks into a
rank-major replica, the ordinary fused kernel, one reduce-scatter of the dense gradient block.
PEER exchange (one NVLink / NVSwitch node, rows <= 128 floats; `exchange='peer'` / `'peer_graph'`): no exchange buffers at all.
Every rank maps the allocations behind its peers' arenas (CUDA IPC, hsk_peer_export / _open); hsk_mf_train_fused_peer reads
each item row from its owner's HBM and reduces the row / bias gradients into the owner's gradient arena over NVLink
(red.relaxed.sys), writing the owner's row stamps; two hsk_peer_barrier launches bracket it (all parameters in place /
all reductions landed).  cfg4, 8 GPUs: 0.96 ms per step against 1.34 ms for the sparse exchange.
Evaluation (`evaluate`; `evaluate_replicated` = user-parallel over a gathered replica; `evaluate_streamed` = shards read in
place through peer mappings): user rows of a round are all-gathered, every rank scores them against its item shard (hsk_eval_topk /
hsk_eval_topk_tc + hsk_rescore_topk with id_offset = rank, id_stride = G), the per-shard top-k lists are exchanged
(all-to-all) so that each rank merges (hsk_topk_merge) and scores the metrics of ITS users; the collectives of round
r + 1 / r - 1 run on a second stream under the scoring of round r; per-group sums are all-reduced once per sweep.

The index bookkeeping is device-agnostic torch code, the arithmetic goes through an `ops` object: `CudaOps` (the
kernels) in production; the world-size-2 gloo tests on CPU plug in a torch reference to check the routing.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.distributed as dist

from hassaku_b200 import _C, determinism, nvtx
from hassaku_b200.algorithms.sgd_alg import ArenaLayout


class ShardSpec:
    def __init__(self, world: int, rank: int, n_users: int, n_items: int):
        self.world, self.rank, self.n_users, self.n_items = world, rank, n_users, n_items
        self.n_local_users = len(range(rank, n_users, world))
        self.n_local_items = len(range(rank, n_items, world))

    def local_count(self, n: int, rank: int) -> int:
        return len(range(rank, n, self.world))


def exchange_capacity(n_slots: int, n_items: int, world: int) -> int:
    """Rows per owner of the sparse exchange's fixed-capacity buffers: the expected number of distinct items among
    n_slots uniform draws (an upper bound for popularity-skewed positives), per owner, + 10 % + 256."""
    cap = math.ceil(n_items / world)
    expect = n_items * (1.0 - math.exp(-n_slots / n_items)) / world
    return int(min(cap, math.ceil(1.10 * expect) + 256))


class CudaOps:
    """The arithmetic / routing of the sharded step on the sm_100a kernels."""

    def __init__(self, status: Optional[torch.Tensor] = None):
        self.status = status

    def local_index(self, idx: torch.Tensor, world: int, rank_stride: int) -> torch.Tensor:
        return _C.shard_local_index(idx.contiguous(), world, rank_stride)

    def route(self, i_global, n_items, world, capq, ld, req_rows, req_count, compact_idx, scratch):
        _C.route_items(i_global, n_items, world, capq, ld, req_rows, req_count, compact_idx, scratch, self.status)

    def pack(self, V2d, Ib, rows, world, capq, out):
        _C.shard_pack(V2d, Ib, rows, world, capq, out, self.status)

    def unpack_add(self, inp, rows, world, capq, gV2d, gIb, stamps, step, step_dev):
        _C.shard_unpack_add(inp, rows, world, capq, gV2d, gIb, stamps, step, step_dev, self.status)

    def unpack_ordered(self, inp, rows, world, capq, gV2d, gIb, stamps, step, step_dev):
        _C.shard_unpack_add(inp, rows, world, capq, gV2d, gIb, stamps, step, step_dev, self.status, ordered=True)

    def mark_rows(self, idx, n_rows, stamps, step, step_dev):
        _C.mark_rows(idx, n_rows, stamps, step, step_dev)

    def train_fused(self, lay: ArenaLayout, arena, g_arena, Vc, Ibc, gVc, gIbc, u_local, compact_idx, B_global, kind, shift,
                    loss_accum):
        Uw, _, Ub, _, Gb = lay.views(arena)
        gU, _, gUb, _, gGb = lay.views(g_arena)
        t = _C.make_tables(Uw, Vc[:, :lay.d], Ub, Ibc, Gb, lay.d)
        g = _C.make_tables(gU, gVc[:, :lay.d], gUb, gIbc, gGb, lay.d)
        _C.mf_train_fused_n(t, g, u_local, compact_idx, B_global, kind, shift, loss_accum, self.status)

    def det_scratch_bytes(self, B, N1, ld):
        return _C.det_scratch_bytes(B, N1, ld)

    def train_fused_det(self, lay: ArenaLayout, arena, g_arena, Vc, Ibc, gVc, gIbc, u_local, compact_idx, B_global, kind, shift,
                        loss_accum, scratch, dscores_out=None):
        """train_fused in the fixed order of deterministic mode (hsk_mf_train_fused_det_n): touched rows are STORED."""
        Uw, _, Ub, _, Gb = lay.views(arena)
        gU, _, gUb, _, gGb = lay.views(g_arena)
        t = _C.make_tables(Uw, Vc[:, :lay.d], Ub, Ibc, Gb, lay.d)
        g = _C.make_tables(gU, gVc[:, :lay.d], gUb, gIbc, gGb, lay.d)
        _C.mf_train_fused_det(t, g, u_local, compact_idx, kind, shift, loss_accum, scratch, dscores_out=dscores_out,
                              status=self.status, B_global=B_global)

    def train_fused_peer(self, lay: ArenaLayout, arena, g_arena, peers, n_items_global, u_local, i_global, B_global, kind, shift,
                         loss_accum, step, step_dev):
        t, g = lay.tables(arena), lay.tables(g_arena)
        t.n_items = g.n_items = n_items_global      # i_global holds GLOBAL ids; the item tables come from `peers`
        _C.mf_train_fused_peer(t, g, peers, u_local, i_global, B_global, kind, shift, loss_accum, step, step_dev, self.status)

    def adamw(self, arena, m, v, g, segments, lr, wd, t, decoupled=True, consts_dev=None, step_dev=None):
        """torch.optim.AdamW / Adam over the local arena; `segments` = row ranges whose untouched rows skip the gradient
        traffic (see hsk_adamw_dense_rows); consts_dev / step_dev: graph mode."""
        _C.adamw_dense_rows(arena, m, v, g, segments, lr, 0.9, 0.999, 1e-8, wd, t, arith=0, adam_l2=not decoupled,
                            consts_dev=consts_dev, step_dev=step_dev)


class ShardedMF:
    """The local shard of an SGDMatrixFactorization plus its optimizer state."""

    CONST_TABLE_STEPS = 32768   # AdamW scalars of the next steps in device memory (1 MB): refills practically never happen

    def __init__(self, n_users: int, n_items: int, d: int, use_user_bias=False, use_item_bias=False, use_global_bias=False,
                 world: Optional[int] = None, rank: Optional[int] = None, device='cuda', ops=None, group=None):
        world = dist.get_world_size(group) if world is None else world
        rank = dist.get_rank(group) if rank is None else rank
        if n_users < world or n_items < world:
            # a rank without a user or an item row would hand the kernels empty tables
            raise ValueError(f'ShardedMF needs at least one user row and one item row per rank: n_users ({n_users}) and '
                             f'n_items ({n_items}) must be >= world ({world})')
        self.spec = ShardSpec(world, rank, n_users, n_items)
        self.d, self.group, self.device = d, group, torch.device(device)
        self.flags = (use_user_bias, use_item_bias, use_global_bias)
        self.layout = ArenaLayout(self.spec.n_local_users, self.spec.n_local_items, d, *self.flags)
        self.arena = torch.zeros(self.layout.n_total, dtype=torch.float32, device=self.device)
        self.m = torch.zeros_like(self.arena)
        self.v = torch.zeros_like(self.arena)
        self.g = torch.zeros_like(self.arena)
        self.t = 0
        cuda = self.device.type == 'cuda'
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device) if cuda else None
        self.ops = ops if ops is not None else CudaOps(self.status)
        self.loss_accum = torch.zeros(1, dtype=torch.float64, device=self.device)
        self.stamp_users = torch.zeros(max(self.spec.n_local_users, 1), dtype=torch.uint8, device=self.device)
        self.stamp_items = torch.zeros(max(self.spec.n_local_items, 1), dtype=torch.uint8, device=self.device)
        self._sparse, self._dense, self._graphs = {}, None, {}
        self._ordered = {}
        self._rank_ordered_loss = False     # set by the ordered exchange: pop_loss sums the ranks' losses in rank order
        self._peer = None
        self._ipc = {}          # (rank, IPC handle) -> base address here of a peer's allocation (opened once, closed in close())

    # ---- collectives (skipped at world 1, where every exchange is the identity) ----
    def _a2a(self, out: torch.Tensor, inp: torch.Tensor):
        if self.spec.world == 1:
            out.copy_(inp)
        else:
            dist.all_to_all_single(out, inp, group=self.group)

    def _all_gather(self, out: torch.Tensor, inp: torch.Tensor):
        if self.spec.world == 1:
            out.view(-1).copy_(inp.view(-1))
        else:
            dist.all_gather_into_tensor(out, inp, group=self.group)

    def _all_reduce(self, t: torch.Tensor, op=None):
        if self.spec.world > 1:
            dist.all_reduce(t, op=op if op is not None else dist.ReduceOp.SUM, group=self.group)

    def _rank_ordered_sum(self, t: torch.Tensor):
        """t = the ranks' values of t added in rank order, starting from rank 0's (all-gather, then G - 1 adds): the same
        bits on every run, where an all-reduce's summation order depends on the collective's algorithm."""
        G = self.spec.world
        if G == 1:
            return
        every = torch.empty((G,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        self._all_gather(every, t.contiguous())
        t.copy_(every[0])
        for q in range(1, G):
            t.add_(every[q])

    def _reduce_metric_sums(self, evaluator):
        """The evaluator's per-rank metric sums and counts summed over the ranks; under torch.use_deterministic_algorithms
        the floating-point sums are added in rank order (every rank's evaluator already sums in a fixed order there)."""
        det = determinism.enabled()
        for name in ('_sums', '_counts', '_hit_sums'):
            x = getattr(evaluator, name, None)
            if x is None:
                continue
            if det and x.is_floating_point():
                self._rank_ordered_sum(x)
            else:
                self._all_reduce(x)

    def _reduce_scatter(self, out: torch.Tensor, inp: torch.Tensor):
        if self.spec.world == 1:
            out.view(-1).copy_(inp.view(-1))
        elif dist.get_backend(self.group) == 'nccl':
            dist.reduce_scatter_tensor(out, inp, group=self.group)
        else:  # gloo (CPU tests) has no reduce-scatter
            dist.all_reduce(inp, group=self.group)
            n = out.numel()
            out.copy_(inp.view(-1)[self.spec.rank * n:(self.spec.rank + 1) * n].view_as(out))

    # ---- state in / out ----
    def load_full_state_dict(self, sd: Dict[str, torch.Tensor]):
        """Take this rank's rows of a full (reference-format) state_dict."""
        G, r = self.spec.world, self.spec.rank
        Uw, Vw, Ub, Ib, Gb = self.layout.views(self.arena)
        with torch.no_grad():
            Uw.copy_(sd['user_embeddings.weight'][r::G].to(self.device))
            Vw.copy_(sd['item_embeddings.weight'][r::G].to(self.device))
            if Ub is not None:
                Ub.copy_(sd['user_bias.weight'][r::G].to(self.device))
            if Ib is not None:
                Ib.copy_(sd['item_bias.weight'][r::G].to(self.device))
            if Gb is not None:
                Gb.copy_(sd['global_bias'].to(self.device))

    def full_state_dict(self, to_cpu: bool = True) -> Dict[str, torch.Tensor]:
        """All-gather the shards into a full state_dict (checkpoint in the reference's format; parity tests)."""
        G = self.spec.world
        Uw, Vw, Ub, Ib, Gb = self.layout.views(self.arena)

        def gather(local, n_total):
            width = local.shape[1]
            cap = math.ceil(n_total / G)
            buf = torch.zeros((cap, width), dtype=torch.float32, device=self.device)
            buf[:local.shape[0]] = local
            allb = torch.empty((G * cap, width), dtype=torch.float32, device=self.device)
            self._all_gather(allb, buf)
            full = torch.empty((n_total, width), dtype=torch.float32, device=self.device)
            for q in range(G):
                full[q::G] = allb[q * cap:q * cap + self.spec.local_count(n_total, q)]
            return full.cpu() if to_cpu else full

        sd = {'user_embeddings.weight': gather(Uw, self.spec.n_users), 'item_embeddings.weight': gather(Vw, self.spec.n_items)}
        if Ub is not None:
            sd['user_bias.weight'] = gather(Ub, self.spec.n_users)
        if Ib is not None:
            sd['item_bias.weight'] = gather(Ib, self.spec.n_items)
        if Gb is not None:
            sd['global_bias'] = Gb.detach().cpu().clone() if to_cpu else Gb.detach().clone()
        return sd

    # ---- helpers ----
    def _table2d(self, arena, which: str):
        lay = self.layout
        off, rows = (lay.off_V, lay.n_items) if which == 'V' else (lay.off_U, lay.n_users)
        return arena[off:off + rows * lay.ld].view(rows, lay.ld)

    def _segments(self, users: bool, items: bool):
        lay, segs = self.layout, []
        if users and lay.n_users > 0:
            segs.append((lay.off_U, lay.n_users, lay.ld, self.stamp_users))
        if items and lay.n_items > 0:
            segs.append((lay.off_V, lay.n_items, lay.ld, self.stamp_items))
        return segs

    # ---- SPARSE exchange: fixed-capacity padded all-to-alls, device-side routing ----
    def _sparse_buffers(self, n_slots: int, capq: Optional[int]):
        return self._exchange_buffers(self._sparse, n_slots, capq)

    def _exchange_buffers(self, store: dict, n_slots: int, capq: Optional[int], shape=None):
        """The sparse exchange's buffers for one batch shape (`store`: the buffer sets of one exchange).  `shape` (B, N1):
        the ordered exchange's set, which also holds the compact index and the deterministic step's scratch — a captured
        graph holds their addresses, so a graph of an evicted set is dropped with it."""
        G, lay, dev = self.spec.world, self.layout, self.device
        capq = capq or exchange_capacity(n_slots, self.spec.n_items, G)
        key = (n_slots, capq) if shape is None else (tuple(shape), capq)
        if key not in store:
            if len(store) >= 2:      # a new batch shape (e.g. the epoch's tail batch): keep at most two sets of buffers
                old = next(iter(store))
                store.pop(old)
                if shape is not None:
                    for gk in [k for k in self._graphs if k[0] == 'ordered' and k[1] == old[0]]:
                        self._drop_graph(gk)
            ld = lay.ld
            br = capq + math.ceil(capq / ld)                       # == hsk_shard_block_rows(capq, ld)
            z = lambda shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device=dev)
            n_scr = _C.route_scratch_bytes(self.spec.n_items, G) if dev.type == 'cuda' else 16
            grads = z(G * br * ld + G * br)                         # [gVc | gIbc]: one memset per step
            store[key] = {
                'capq': capq, 'br': br,
                'req_rows': z((G, capq), torch.int32), 'req_count': z(G, torch.int32),
                'recv_rows': z((G, capq), torch.int32), 'scratch': z(n_scr, torch.uint8),
                'send': z((G, br, ld)), 'Vc': z((G * br, ld)), 'Ibc': z(G * br),
                'grads': grads, 'gVc': grads[:G * br * ld].view(G * br, ld), 'gIbc': grads[G * br * ld:],
                'recv_g': z((G, br, ld)),
            }
            if shape is not None:
                B, N1 = shape
                store[key]['compact_idx'] = z((B, N1), torch.int64)
                store[key]['det'] = z(max(self.ops.det_scratch_bytes(B, N1, ld), 16), torch.uint8)
        return store[key]

    def _sparse_body(self, u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled, capq=None, consts_dev=None,
                     step_dev=None):
        G, lay = self.spec.world, self.layout
        ld = lay.ld
        S = self._sparse_buffers(i_global.numel(), capq)
        capq, br = S['capq'], S['br']
        _, _, _, Ib, _ = lay.views(self.arena)
        has_ib = Ib is not None
        step = self.t + 1
        compact_idx = torch.empty_like(i_global)
        # 1-2. who needs which rows; tell the owners
        self.ops.route(i_global, self.spec.n_items, G, capq, ld, S['req_rows'], S['req_count'], compact_idx, S['scratch'])
        self._a2a(S['recv_rows'], S['req_rows'])
        # 3. owners pack rows (+ biases in the block's tail rows) and send them back
        self.ops.pack(self._table2d(self.arena, 'V'), Ib.view(-1) if has_ib else None, S['recv_rows'], G, capq, S['send'])
        self._a2a(S['Vc'].view(G, br, ld), S['send'])
        if has_ib:
            S['Ibc'].view(G, br)[:, :capq] = S['Vc'].view(G, br * ld)[:, capq * ld:capq * ld + capq]
        # 4. local compute on (user shard, compact item table)
        S['grads'].zero_()
        u_local = self.ops.local_index(u_global, G, 0)
        self.ops.mark_rows(u_local, lay.n_users, self.stamp_users, step, step_dev)
        self.ops.train_fused(lay, self.arena, self.g, S['Vc'], S['Ibc'] if has_ib else None, S['gVc'],
                             S['gIbc'] if has_ib else None, u_local, compact_idx, B_global, _C.LOSS_KINDS[loss_kind], neg_shift,
                             self.loss_accum)
        # 5. gradients home (bias gradients ride in the tail rows of the same blocks)
        if has_ib:
            S['gVc'].view(G, br * ld)[:, capq * ld:capq * ld + capq] = S['gIbc'].view(G, br)[:, :capq]
        self._a2a(S['recv_g'], S['gVc'].view(G, br, ld))
        gIb = lay.views(self.g)[3]
        self.ops.unpack_add(S['recv_g'], S['recv_rows'], G, capq, self._table2d(self.g, 'V'),
                            gIb.view(-1) if gIb is not None else None, self.stamp_items, step, step_dev)
        gGb = lay.views(self.g)[4]
        if gGb is not None:
            self._all_reduce(gGb)   # the global bias is replicated: every rank applies the summed gradient
        # 6. optimizer on the local shard
        self.ops.adamw(self.arena, self.m, self.v, self.g, self._segments(True, True), lr, wd, step, decoupled,
                       consts_dev=consts_dev, step_dev=step_dev)

    def train_step(self, u_global: torch.Tensor, i_global: torch.Tensor, B_global: int, loss_kind: str, neg_shift: float,
                   lr: float, wd: float, decoupled: bool = True, capq: Optional[int] = None):
        """u_global int64 [B_r] (all owned by this rank: u % G == rank), i_global int64 [B_r, 1+N] global item ids."""
        self._sparse_body(u_global, i_global.contiguous(), B_global, loss_kind, neg_shift, lr, wd, decoupled, capq)
        self.t += 1

    # ---- ORDERED exchange: the sparse exchange with every cross-row and cross-rank float reduction in a fixed order
    # (order contract of the sharded step, include/hassaku_b200.h): bitwise reproducible at a fixed world size ----
    def _ordered_body(self, u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled, capq=None, consts_dev=None,
                      step_dev=None):
        """_sparse_body with hsk_mf_train_fused_det_n instead of the atomic fused kernel, hsk_shard_unpack_ordered instead
        of the atomic unpack-add, and the global-bias gradient summed in rank order instead of by an all-reduce."""
        G, lay = self.spec.world, self.layout
        ld = lay.ld
        S = self._exchange_buffers(self._ordered, i_global.numel(), capq, shape=i_global.shape)
        capq, br = S['capq'], S['br']
        _, _, _, Ib, _ = lay.views(self.arena)
        has_ib = Ib is not None
        step = self.t + 1
        self._rank_ordered_loss = True
        compact_idx = S['compact_idx']
        self.ops.route(i_global, self.spec.n_items, G, capq, ld, S['req_rows'], S['req_count'], compact_idx, S['scratch'])
        self._a2a(S['recv_rows'], S['req_rows'])
        self.ops.pack(self._table2d(self.arena, 'V'), Ib.view(-1) if has_ib else None, S['recv_rows'], G, capq, S['send'])
        self._a2a(S['Vc'].view(G, br, ld), S['send'])
        if has_ib:
            S['Ibc'].view(G, br)[:, :capq] = S['Vc'].view(G, br * ld)[:, capq * ld:capq * ld + capq]
        S['grads'].zero_()
        u_local = self.ops.local_index(u_global, G, 0)
        self.ops.mark_rows(u_local, lay.n_users, self.stamp_users, step, step_dev)
        self.ops.train_fused_det(lay, self.arena, self.g, S['Vc'], S['Ibc'] if has_ib else None, S['gVc'],
                                 S['gIbc'] if has_ib else None, u_local, compact_idx, B_global, _C.LOSS_KINDS[loss_kind],
                                 neg_shift, self.loss_accum, S['det'])
        if has_ib:
            S['gVc'].view(G, br * ld)[:, capq * ld:capq * ld + capq] = S['gIbc'].view(G, br)[:, :capq]
        self._a2a(S['recv_g'], S['gVc'].view(G, br, ld))
        gIb = lay.views(self.g)[3]
        self.ops.unpack_ordered(S['recv_g'], S['recv_rows'], G, capq, self._table2d(self.g, 'V'),
                                gIb.view(-1) if gIb is not None else None, self.stamp_items, step, step_dev)
        gGb = lay.views(self.g)[4]
        if gGb is not None:
            self._rank_ordered_sum(gGb)
        self.ops.adamw(self.arena, self.m, self.v, self.g, self._segments(True, True), lr, wd, step, decoupled,
                       consts_dev=consts_dev, step_dev=step_dev)

    def train_step_ordered(self, u_global: torch.Tensor, i_global: torch.Tensor, B_global: int, loss_kind: str,
                           neg_shift: float, lr: float, wd: float, decoupled: bool = True, capq: Optional[int] = None):
        """The step with the ORDERED exchange (see _ordered_body): the same bits on every run at a fixed world size, with or
        without torch.use_deterministic_algorithms."""
        self._ordered_body(u_global, i_global.contiguous(), B_global, loss_kind, neg_shift, lr, wd, decoupled, capq)
        self.t += 1

    def train_step_ordered_graphed(self, *a, capq=None):
        return self._graphed(self._ordered_body, 'ordered', *a, capq)

    # ---- DENSE exchange: when the batch touches (nearly) every item anyway ----
    def _dense_buffers(self):
        """Send / replica buffers of the dense exchange.  One rank's block is [capP, ld] floats: rows [0, cap) are its item
        rows (cap = ceil(n_items / G), unused rows zero), rows [cap, capP) hold its cap item biases flat - so ONE
        all-gather moves rows and biases, and ONE reduce-scatter brings back both gradients.  The fused kernel indexes
        the replica as a [G * capP, ld] table (row of item i = (i % G) * capP + i // G) and needs the biases under the
        same index, hence the compact `Ib` / `gIb` vectors of G * capP floats filled / drained by one strided copy."""
        if self._dense is None:
            G, lay = self.spec.world, self.layout
            cap = math.ceil(self.spec.n_items / G)
            capP = cap + math.ceil(cap / lay.ld)
            z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=self.device)
            grads = z(G * capP * lay.ld + G * capP)          # [gV replica | gIb compact]: one memset per step
            self._dense = {'cap': cap, 'capP': capP, 'V': z(G * capP, lay.ld), 'Ib': z(G * capP),
                           'grads': grads, 'gV': grads[:G * capP * lay.ld].view(G * capP, lay.ld),
                           'gIb': grads[G * capP * lay.ld:], 'send': z(capP, lay.ld), 'recv': z(capP, lay.ld)}
        return self._dense

    def _dense_body(self, u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled, capq=None, consts_dev=None,
                    step_dev=None):
        """All-gather of the item shards into the rank-major replica, the ordinary fused kernel on it, reduce-scatter of
        the dense item gradient to the owners.  No dedupe, no host sync, fixed shapes: 2 collectives, 1 memset, 2 index
        kernels, 4 small copies around the fused kernel."""
        G, lay = self.spec.world, self.layout
        ld, nl = lay.ld, lay.n_items
        D = self._dense_buffers()
        cap, capP = D['cap'], D['capP']
        _, _, _, Ib, _ = lay.views(self.arena)
        has_ib = Ib is not None
        step = self.t + 1
        D['send'][:nl] = self._table2d(self.arena, 'V')
        if has_ib:
            D['send'].view(-1)[cap * ld:cap * ld + nl] = Ib.view(-1)
        self._all_gather(D['V'], D['send'])
        if has_ib:
            D['Ib'].view(G, capP)[:, :cap] = D['V'].view(G, capP * ld)[:, cap * ld:cap * ld + cap]
        rows = self.ops.local_index(i_global, G, capP)
        u_local = self.ops.local_index(u_global, G, 0)
        sparse_users = 4 * u_global.numel() <= lay.n_users
        if sparse_users:
            self.ops.mark_rows(u_local, lay.n_users, self.stamp_users, step, step_dev)
        D['grads'].zero_()
        self.ops.train_fused(lay, self.arena, self.g, D['V'], D['Ib'] if has_ib else None, D['gV'],
                             D['gIb'] if has_ib else None, u_local, rows, B_global,
                             _C.LOSS_KINDS[loss_kind], neg_shift, self.loss_accum)
        if has_ib:
            D['gV'].view(G, capP * ld)[:, cap * ld:cap * ld + cap] = D['gIb'].view(G, capP)[:, :cap]
        self._reduce_scatter(D['recv'], D['gV'])
        self._table2d(self.g, 'V').add_(D['recv'][:nl])
        if has_ib:
            lay.views(self.g)[3].view(-1).add_(D['recv'].view(-1)[cap * ld:cap * ld + nl])
        gGb = lay.views(self.g)[4]
        if gGb is not None:
            self._all_reduce(gGb)
        self.ops.adamw(self.arena, self.m, self.v, self.g, self._segments(sparse_users, False), lr, wd, step, decoupled,
                       consts_dev=consts_dev, step_dev=step_dev)

    # ---- PEER exchange: no exchange buffers at all — the step kernel reads the item rows from, and reduces their
    # gradients into, the owners' memory over NVLink ----
    PEER_MAX_LD = 128
    peer_barrier = 'kernel'      # 'kernel': hsk_peer_barrier (flags in peer memory); 'nccl': a 4-byte all-reduce

    def peer_supported(self) -> bool:
        return self.device.type == 'cuda' and self.spec.world <= _C.MAX_PEERS and self.layout.ld <= self.PEER_MAX_LD

    def _peer_setup(self):
        """Once: every rank exports the allocations behind its parameter arena, gradient arena and item stamps (CUDA IPC),
        maps its peers' and builds the table of item-shard addresses the kernel indexes by owner."""
        if self._peer is not None:
            return self._peer
        G, r, lay = self.spec.world, self.spec.rank, self.layout
        if not self.peer_supported():
            raise _C.HskError(f'the peer exchange needs CUDA, at most {_C.MAX_PEERS} ranks on one node and rows of at most '
                              f'{self.PEER_MAX_LD} floats (world {G}, ld {lay.ld}): use the sparse / dense exchange')
        mine = {'off_V': lay.off_V, 'off_Ib': lay.off_Ib}
        flags = torch.zeros(_C.MAX_PEERS, dtype=torch.int32, device=self.device)      # barrier arrival flags, written by the peers
        local = (self.arena, self.g, self.stamp_items, flags)
        if G > 1:
            import socket
            mine['host'] = socket.gethostname()
            try:
                mine['exports'] = [_C.peer_export(t) for t in local]
            except _C.HskError as ex:        # e.g. an allocator that cannot export (expandable segments): tell the peers
                mine['error'] = str(ex)
            every = [None] * G
            dist.all_gather_object(every, mine, group=self.group)
            errs = [f"rank {q}: {e['error']}" for q, e in enumerate(every) if 'error' in e]
            if errs:
                raise _C.HskError('the peer exchange is not available (CUDA IPC export failed: ' + '; '.join(errs) +
                                  '): use the sparse / dense exchange')
            if len({e['host'] for e in every}) != 1:
                raise _C.HskError('the peer exchange maps the other ranks\' memory (CUDA IPC over NVLink): all ranks must run on '
                                  'one node — use the sparse / dense exchange across nodes')
        else:
            every = [mine]
        opened = self._ipc

        def addr(q, which):          # address in THIS process of tensor `which` of rank q
            if q == r:
                return local[which].data_ptr()
            handle, off = every[q]['exports'][which]
            if (q, handle) not in opened:
                opened[(q, handle)] = _C.peer_open(handle, self.device)
            return opened[(q, handle)] + off

        has_ib = lay.off_Ib >= 0
        failure = None
        try:
            V = [addr(q, 0) + 4 * every[q]['off_V'] for q in range(G)]
            gV = [addr(q, 1) + 4 * every[q]['off_V'] for q in range(G)]
            Ib = [addr(q, 0) + 4 * every[q]['off_Ib'] for q in range(G)] if has_ib else None
            gIb = [addr(q, 1) + 4 * every[q]['off_Ib'] for q in range(G)] if has_ib else None
            st = [addr(q, 2) for q in range(G)]
            fl = [addr(q, 3) for q in range(G)]
        except _C.HskError as ex:
            failure = str(ex)
        if G > 1:       # every rank learns whether EVERY rank could map its peers (same collectives on every path)
            ok = torch.tensor([0 if failure else 1], dtype=torch.int32, device=self.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if int(ok.item()) == 0:
                raise _C.HskError('the peer exchange is not available (mapping a peer\'s memory failed' +
                                  (f': {failure}' if failure else ' on another rank') + '): use the sparse / dense exchange')
        elif failure:
            raise _C.HskError(failure)
        self._peer = {'items': _C.make_peer_items(V, gV, Ib, gIb, st), 'opened': opened,
                      'bar': torch.zeros(1, dtype=torch.float32, device=self.device),
                      'flags': flags, 'flag_table': _C.make_peer_flags(fl, r),
                      'epoch': torch.zeros(1, dtype=torch.int32, device=self.device)}
        if G > 1:
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)       # every rank's flags are zero and mapped before the first arrival is written
        return self._peer

    def _barrier(self):
        """Stream-ordered cross-rank barrier (graph-capturable): the work every rank enqueued before it is complete before
        anything enqueued after it starts on any rank."""
        if self.spec.world > 1:
            if self.peer_barrier == 'kernel':
                _C.peer_barrier(self._peer['flag_table'], self._peer['epoch'], self.status)
            else:
                dist.all_reduce(self._peer['bar'], group=self.group)

    def _peer_body(self, u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled, capq=None, consts_dev=None,
                   step_dev=None):
        P = self._peer_setup()
        G, lay = self.spec.world, self.layout
        step = self.t + 1
        self._barrier()      # every rank's parameters (previous AdamW, a load, a restore) and zeroed gradients are in place
        u_local = self.ops.local_index(u_global, G, 0)
        self.ops.mark_rows(u_local, lay.n_users, self.stamp_users, step, step_dev)
        self.ops.train_fused_peer(lay, self.arena, self.g, P['items'], self.spec.n_items, u_local, i_global, B_global,
                                  _C.LOSS_KINDS[loss_kind], neg_shift, self.loss_accum, step, step_dev)
        self._barrier()      # every rank's gradient contributions and stamps have landed at their owners
        gGb = lay.views(self.g)[4]
        if gGb is not None:
            self._all_reduce(gGb)
        self.ops.adamw(self.arena, self.m, self.v, self.g, self._segments(True, True), lr, wd, step, decoupled,
                       consts_dev=consts_dev, step_dev=step_dev)

    def train_step_peer(self, u_global: torch.Tensor, i_global: torch.Tensor, B_global: int, loss_kind: str, neg_shift: float,
                        lr: float, wd: float, decoupled: bool = True, capq=None):
        """The step with the PEER exchange (see _peer_body): 2 barriers + 4 kernels, nothing staged."""
        self._peer_body(u_global, i_global.contiguous(), B_global, loss_kind, neg_shift, lr, wd, decoupled)
        self.t += 1

    def train_step_peer_graphed(self, *a, capq=None):
        return self._graphed(self._peer_body, 'peer', *a, capq)

    def train_step_dense(self, u_global: torch.Tensor, i_global: torch.Tensor, B_global: int, loss_kind: str,
                         neg_shift: float, lr: float, wd: float, decoupled: bool = True, capq=None):
        """Same step with a DENSE exchange (see _dense_body).  The right choice when B (N + 1) >> n_items (cfg2: 418 k
        slots on 3 706 items, every row is requested by every rank each step anyway)."""
        self._dense_body(u_global, i_global.contiguous(), B_global, loss_kind, neg_shift, lr, wd, decoupled)
        self.t += 1

    # ---- either step as ONE CUDA graph (fixed shapes): removes the launches / collectives worth of host latency ----
    def _fill_const_table(self, gs, lr, wd):
        host = torch.empty((self.CONST_TABLE_STEPS, 8), dtype=torch.float32).pin_memory()
        for j in range(self.CONST_TABLE_STEPS):
            _C.adamw_consts(lr, 0.9, 0.999, 1e-8, wd, self.t + 1 + j, host[j])
        gs['table'].copy_(host)
        gs['step_idx'].zero_()
        gs['step_dev'].fill_(self.t + 1)
        gs['table_base_t'] = self.t

    def _graphed(self, body, name, u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled, capq):
        """`body` captured once per (exchange, batch shape, hyper-parameters) and replayed.  The per-step AdamW scalars
        come from a device table of the next CONST_TABLE_STEPS steps indexed by a device-side step counter, the row
        stamps from the device-side 1-based step count: a replay needs no host-computed kernel argument."""
        key = (name, tuple(i_global.shape), B_global, loss_kind, float(neg_shift), float(lr), float(wd), bool(decoupled), capq)
        gs = self._graphs.get(key)
        if gs is None:
            if len(self._graphs) >= 3:
                self._drop_graph(next(iter(self._graphs)))
            dev = self.device
            gs = {'u': torch.empty_like(u_global, device=dev), 'i': torch.empty_like(i_global, device=dev),
                  'table': torch.empty((self.CONST_TABLE_STEPS, 8), dtype=torch.float32, device=dev),
                  'consts': torch.empty(8, dtype=torch.float32, device=dev),
                  'step_idx': torch.zeros(1, dtype=torch.int64, device=dev),
                  'step_dev': torch.zeros(1, dtype=torch.int64, device=dev)}
            self._fill_const_table(gs, lr, wd)
            gs['u'].copy_(u_global); gs['i'].copy_(i_global)
            # NCCL channels / buffers of this body must exist before capture: run it once eagerly on a scratch copy of the
            # state that the step mutates (parameters, optimizer state, loss, stamps are restored afterwards)
            saved = [x.clone() for x in (self.arena, self.m, self.v, self.g, self.loss_accum, self.stamp_users, self.stamp_items)]
            body(gs['u'], gs['i'], B_global, loss_kind, neg_shift, lr, wd, decoupled, capq)
            for dst, src in zip((self.arena, self.m, self.v, self.g, self.loss_accum, self.stamp_users, self.stamp_items), saved):
                dst.copy_(src)
            del saved
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                torch.index_select(gs['table'], 0, gs['step_idx'], out=gs['consts'].view(1, 8))
                body(gs['u'], gs['i'], B_global, loss_kind, neg_shift, lr, wd, decoupled, capq, consts_dev=gs['consts'],
                     step_dev=gs['step_dev'])
                gs['step_idx'].add_(1)
                gs['step_dev'].add_(1)
            gs['graph'] = graph
            self._graphs[key] = gs
        if self.t - gs['table_base_t'] >= self.CONST_TABLE_STEPS or int(gs.get('expect_t', self.t)) != self.t:
            torch.cuda.current_stream().synchronize()   # another graph / an eager step advanced t: re-base the device counters
            self._fill_const_table(gs, lr, wd)
        gs['u'].copy_(u_global, non_blocking=True)
        gs['i'].copy_(i_global, non_blocking=True)
        gs['graph'].replay()
        self.t += 1
        gs['expect_t'] = self.t

    def _drop_graph(self, key):
        torch.cuda.synchronize()
        self._graphs.pop(key, None)

    def train_step_graphed(self, *a, capq=None):
        return self._graphed(self._sparse_body, 'sparse', *a, capq)

    def train_step_dense_graphed(self, *a, capq=None):
        return self._graphed(self._dense_body, 'dense', *a, capq)

    def close(self):
        """Drop the captured CUDA graphs (they hold NCCL work): call before dist.destroy_process_group(), which
        otherwise blocks."""
        if self.device.type == 'cuda':
            torch.cuda.synchronize()
        self._graphs = {}
        import gc
        gc.collect()
        if self.device.type == 'cuda':
            torch.cuda.synchronize()
        if self._ipc:
            if self.spec.world > 1:
                dist.barrier(group=self.group)      # no peer is still inside a kernel that addresses this rank's memory
            for base in self._ipc.values():
                _C.peer_close(base)
            self._ipc = {}
        self._peer = None

    def step(self, u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled=True, exchange='auto', capq=None):
        """Dispatch on the expected fraction of distinct items: dense exchange when the batch covers the item table.
        `exchange='ordered'` / `'ordered_graph'` is the deterministic step (bitwise reproducible at a fixed world size);
        every other exchange reduces gradients from several ranks with floating-point atomics, so it raises under
        torch.use_deterministic_algorithms(True) (warns under warn_only)."""
        if exchange not in ('ordered', 'ordered_graph'):
            determinism.alert_not_deterministic(f"ShardedMF.step(exchange={exchange!r}; exchange='ordered' is the "
                                                "deterministic one)")
        if exchange in ('auto', 'auto_graph'):
            dense = i_global.numel() >= 2 * self.spec.n_items // self.spec.world
            exchange = ('dense' if dense else 'sparse') + ('_graph' if exchange == 'auto_graph' else '')
        fn = {'dense': self.train_step_dense, 'dense_graph': self.train_step_dense_graphed, 'sparse': self.train_step,
              'sparse_graph': self.train_step_graphed, 'peer': self.train_step_peer,
              'peer_graph': self.train_step_peer_graphed, 'ordered': self.train_step_ordered,
              'ordered_graph': self.train_step_ordered_graphed}[exchange]
        with nvtx.range('hsk.sharded_step'):
            return fn(u_global, i_global, B_global, loss_kind, neg_shift, lr, wd, decoupled, capq=capq)

    def pop_loss(self) -> float:
        """Sum over ranks of the batch-mean loss contributions since the last call (one all-reduce + host sync; after an
        ordered step or under torch.use_deterministic_algorithms an all-gather summed in rank order)."""
        t = self.loss_accum.clone()
        if self._rank_ordered_loss or determinism.enabled():
            self._rank_ordered_sum(t)
        else:
            self._all_reduce(t)
        self.loss_accum.zero_()
        return float(t.item())

    def check_status(self):
        """One host sync: raise if a kernel since the last check met a bad index or an exchange buffer overflowed."""
        if self.status is None:
            return
        st = int(self.status.item())
        if st:
            self.status.zero_()
            what = []
            if st & _C.STATUS_BAD_INDEX:
                what.append('an out-of-range user / item index')
            if st & _C.STATUS_CAPACITY:
                what.append('an overflow of the fixed-capacity exchange buffers (raise capq)')
            if st & _C.STATUS_BARRIER_TIMEOUT:
                what.append('a peer barrier that timed out (a rank is missing or ran a different number of steps)')
            raise _C.HskError(f'rank {self.spec.rank}: the sharded step reported ' + ' and '.join(what or [f'status {st}']))

    def _csr_cache(self, m):
        from hassaku_b200.eval.eval import DeviceCSR
        cache = self.__dict__.setdefault('_csr', {})
        if id(m) not in cache:
            cache[id(m)] = (m, DeviceCSR(m, self.device))   # keep `m` alive so the id stays unique
        return cache[id(m)][1]

    # ---- item-sharded full-rank evaluation ----
    RESCORE_MARGIN = 28

    def evaluate(self, labels_csr, exclude_csr, evaluator, batch_size: int = 8192, precision: str = 'fp32',
                 rescore: bool = True, max_rounds: Optional[int] = None, overlap: bool = True):
        """Every rank evaluates ITS users (u % G == rank) against ALL items; returns the global metric dict on every
        rank.  `labels_csr` / `exclude_csr`: full scipy CSR matrices (global ids) or DeviceCSR.  `batch_size` = users per
        rank and round (a round scores G * batch_size users against the local item shard).  precision 'tf32' / 'bf16':
        tcgen05 scoring; with `rescore` the k + 28 best candidates of the local shard are scored again in fp32
        (hsk_rescore_topk) before the merge, so the merged list is the fp32 list.  `max_rounds` bounds the sweep (bench
        samples).  `overlap`: the collectives of neighbouring rounds run on a second stream under the scoring."""
        from hassaku_b200.eval.eval import DeviceCSR
        if precision not in _C.PRECISIONS:
            raise ValueError(f'eval precision {precision!r} not in {sorted(_C.PRECISIONS)}')
        prec = _C.PRECISIONS[precision]          # 0: fp32-exact SIMT kernel; tf32 / bf16: tcgen05 kernel on the local shard
        G, r, lay, dev = self.spec.world, self.spec.rank, self.layout, self.device
        k = max(evaluator.K_VALUES)
        labels = labels_csr if isinstance(labels_csr, DeviceCSR) else self._csr_cache(labels_csr)
        exclude = exclude_csr if isinstance(exclude_csr, DeviceCSR) else self._csr_cache(exclude_csr)
        cap = math.ceil(self.spec.n_users / G)
        bs = min(batch_size, cap)
        ld = lay.ld
        U2d = self._table2d(self.arena, 'U')
        Uw, Vw, Ub, Ib, Gb = lay.views(self.arena)
        Be = G * bs
        kc = min(128, k + self.RESCORE_MARGIN, lay.n_items) if (prec != 0 and rescore) else k
        do_rescore = kc > k
        # G > 1: re-score AFTER the merge — the shards exchange their low-precision top-kc lists, the owner merges them to the
        # global top-kc, every shard scores in fp32 only the merged candidates it owns (kc / G per user on average instead of
        # kc per user and shard), the owner combines: the fp32 work shards with the items like the scoring itself
        late = do_rescore and G > 1
        if prec == 0:
            scratch = torch.empty(_C.eval_topk_scratch_bytes(Be, lay.n_items, k), dtype=torch.uint8, device=dev)
        else:
            scratch = torch.empty(_C.eval_topk_tc_scratch_bytes(Be, lay.n_items, kc), dtype=torch.uint8, device=dev)
            Vq = _C.pack_rows(Vw.detach(), lay.d, prec)         # the local item shard, packed once per sweep
        f32 = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
        i32 = lambda *shape: torch.empty(shape, dtype=torch.int32, device=dev)
        i64 = lambda *shape: torch.empty(shape, dtype=torch.int64, device=dev)
        # double-buffered per round parity: gathered inputs, local results, received lists
        bufs = [{'rows': f32(bs, ld), 'ubias': f32(bs), 'gids': i64(bs), 'all_rows': f32(Be, ld), 'all_ub': f32(Be),
                 'all_gids': i64(Be), 'safe': i64(Be), 'top_s': f32(Be, k), 'top_i': i32(Be, k),
                 'cand_s': f32(Be, kc) if do_rescore else None, 'cand_i': i32(Be, kc) if do_rescore else None,
                 'recv_s': f32(G, bs, kc if late else k), 'recv_i': i32(G, bs, kc if late else k), 'ms': f32(bs, k), 'mi': i32(bs, k),
                 'mcs': f32(bs, kc) if late else None, 'mci': i32(bs, kc) if late else None,
                 'all_mci': i32(Be, kc) if late else None, 'sc': f32(Be, kc) if late else None,
                 'recv_sc': f32(G, bs, kc) if late else None,
                 'ready': None, 'scored': None, 'merged': None} for _ in range(2)]
        u_rows = torch.arange(Be, dtype=torch.int64, device=dev)
        starts = list(range(0, cap, bs))
        if max_rounds is not None:
            starts = starts[:max_rounds]
        use_streams = overlap and dev.type == 'cuda' and G > 1
        main = torch.cuda.current_stream(dev) if dev.type == 'cuda' else None
        comm = torch.cuda.Stream(device=dev) if use_streams else None
        evaluator._prepare(dev)

        def on_comm():
            return torch.cuda.stream(comm) if use_streams else _NullCtx()

        def gather(j):
            """all-gather the user rows / ids / biases of round j (comm stream)."""
            s, b = starts[j], bufs[j % 2]
            n_mine = max(0, min(bs, lay.n_users - s))                 # my users of this round (may be fewer at the tail)
            with on_comm():
                if use_streams and b['merged'] is not None:
                    comm.wait_event(b['scored'])                      # the buffers' previous round has been consumed
                b['rows'].zero_(); b['ubias'].zero_(); b['gids'].fill_(-1)
                if n_mine > 0:
                    b['rows'][:n_mine] = U2d[s:s + n_mine]
                    b['gids'][:n_mine] = torch.arange(s, s + n_mine, device=dev) * G + r
                    if Ub is not None:
                        b['ubias'][:n_mine] = Ub.view(-1)[s:s + n_mine]
                self._all_gather(b['all_rows'], b['rows'])
                self._all_gather(b['all_gids'], b['gids'])
                if Ub is not None:
                    self._all_gather(b['all_ub'], b['ubias'])
                if use_streams:
                    b['ready'] = comm.record_event()
            b['n_mine'] = n_mine

        def score(j):
            b = bufs[j % 2]
            if use_streams:
                main.wait_event(b['ready'])
                if b['merged'] is not None:
                    main.wait_event(b['merged'])                      # top_s / top_i of round j - 2 have been sent
            torch.where(b['all_gids'] >= 0, b['all_gids'], torch.zeros_like(b['all_gids']), out=b['safe'])
            ub = b['all_ub'] if Ub is not None else None
            t = _C.make_tables(b['all_rows'][:, :lay.d], Vw, ub, Ib, Gb, lay.d)
            if prec == 0:
                _C.eval_topk(t, b['safe'], k, b['top_s'], b['top_i'], scratch, exclude.indptr, exclude.indices, id_offset=r,
                             id_stride=G, status=self.status, u_rows=u_rows, n_users_global=self.spec.n_users)
            else:
                Uq = _C.pack_rows(b['all_rows'][:, :lay.d], lay.d, prec)
                cs, ci = (b['cand_s'], b['cand_i']) if do_rescore else (b['top_s'], b['top_i'])
                _C.eval_topk_tc(Uq, Vq, prec, b['safe'], self.spec.n_users, kc, cs, ci, scratch, Ub=ub, Ib=Ib, Gb=Gb,
                                excl_indptr=exclude.indptr, excl_indices=exclude.indices, id_offset=r, id_stride=G,
                                status=self.status, u_rows=u_rows)
                if do_rescore and not late:
                    _C.rescore_topk(t, u_rows, ci, k, b['top_s'], b['top_i'], id_offset=r, id_stride=G, status=self.status,
                                    cand_scores=cs)
            if use_streams:
                b['scored'] = main.record_event()

        def merge(j):
            """exchange: rank q receives the G partial lists of its bs users; merge; metrics (comm stream)."""
            b = bufs[j % 2]
            with on_comm():
                if use_streams:
                    comm.wait_event(b['scored'])
                if late:
                    self._a2a(b['recv_s'], b['cand_s'].view(G, bs, kc))
                    self._a2a(b['recv_i'], b['cand_i'].view(G, bs, kc))
                    _C.topk_merge(b['recv_s'], b['recv_i'], b['mcs'], b['mci'])          # global top-kc by low-precision score
                    self._all_gather(b['all_mci'], b['mci'])
                    ub = b['all_ub'] if Ub is not None else None
                    t = _C.make_tables(b['all_rows'][:, :lay.d], Vw, ub, Ib, Gb, lay.d)
                    _C.rescore_scores(t, u_rows, b['all_mci'], b['sc'], id_offset=r, id_stride=G, status=self.status)
                    self._a2a(b['recv_sc'], b['sc'].view(G, bs, kc))
                    _C.topk_combine(b['recv_sc'], b['mci'], k, b['ms'], b['mi'], cand_scores=b['mcs'])
                else:
                    self._a2a(b['recv_s'], b['top_s'].view(G, bs, k))
                    self._a2a(b['recv_i'], b['top_i'].view(G, bs, k))
                    _C.topk_merge(b['recv_s'], b['recv_i'], b['ms'], b['mi'])
                if b['n_mine'] > 0:
                    n = b['n_mine']
                    evaluator.eval_batch_topk(b['gids'][:n].contiguous(), b['mi'][:n].contiguous(), labels)
                if use_streams:
                    b['merged'] = comm.record_event()

        if starts:
            gather(0)
        for j in range(len(starts)):
            with nvtx.range('hsk.sharded_eval_round'):
                if j + 1 < len(starts):
                    gather(j + 1)        # comm stream: runs under score(j)
                score(j)
                merge(j)                 # comm stream: runs under score(j + 1)
        if use_streams:
            main.wait_stream(comm)
        # one reduction of the accumulators per sweep
        self._reduce_metric_sums(evaluator)
        return evaluator.get_results()


    def evaluate_replicated(self, labels_csr, exclude_csr, evaluator, batch_size: int = 18944, precision: str = 'fp32',
                            rescore: bool = True, max_users: Optional[int] = None):
        """USER-parallel evaluation: the item shards are all-gathered ONCE per sweep into a full replica on every GPU (cfg5:
        1 GB of fp32 rows + 0.5 GB packed bf16, against 180 GB of HBM), then every rank runs the single-GPU pipeline on ITS
        users against ALL items — no per-round collective, no per-shard top-k, one all-reduce of the metric sums at the end.
        The alternative to `evaluate` (item-sharded scoring + top-k merge, what SURVEY 8e specifies) whenever the item table
        fits one GPU: a shard's top-k scan costs nearly as much for I / G items as for I (the candidate lists' warm-up does
        not shrink with the shard), so item-sharding scales sub-linearly while this mode scales with the users.
        `max_users`: bound on the number of LOCAL users evaluated (bench samples)."""
        from hassaku_b200.eval.eval import DeviceCSR
        if precision not in _C.PRECISIONS:
            raise ValueError(f'eval precision {precision!r} not in {sorted(_C.PRECISIONS)}')
        prec = _C.PRECISIONS[precision]
        G, r, lay, dev = self.spec.world, self.spec.rank, self.layout, self.device
        k = max(evaluator.K_VALUES)
        labels = labels_csr if isinstance(labels_csr, DeviceCSR) else self._csr_cache(labels_csr)
        exclude = exclude_csr if isinstance(exclude_csr, DeviceCSR) else self._csr_cache(exclude_csr)
        I, ld = self.spec.n_items, lay.ld
        Uw, Vw, Ub, Ib, Gb = lay.views(self.arena)
        # full item replica (rows + bias), gathered rank-major and un-interleaved: item i = shard (i % G), row i // G
        cap = math.ceil(I / G)
        send = torch.zeros((cap, ld + 4), dtype=torch.float32, device=dev)
        send[:lay.n_items, :ld] = self._table2d(self.arena, 'V')
        if Ib is not None:
            send[:lay.n_items, ld] = Ib.view(-1)
        allb = torch.empty((G * cap, ld + 4), dtype=torch.float32, device=dev)
        self._all_gather(allb, send)
        Vfull = torch.empty((I, ld), dtype=torch.float32, device=dev)
        Ibfull = torch.empty(I, dtype=torch.float32, device=dev) if Ib is not None else None
        for q in range(G):
            n_q = self.spec.local_count(I, q)
            Vfull[q::G] = allb[q * cap:q * cap + n_q, :ld]
            if Ibfull is not None:
                Ibfull[q::G] = allb[q * cap:q * cap + n_q, ld]
        del allb, send
        n_loc = lay.n_users if max_users is None else min(lay.n_users, max_users)
        bs = max(1, min(batch_size, n_loc))
        kc = min(128, k + self.RESCORE_MARGIN, I) if (prec != 0 and rescore) else k
        U2d = self._table2d(self.arena, 'U')
        t = _C.make_tables(U2d[:, :lay.d], Vfull[:, :lay.d], Ub, Ibfull, Gb, lay.d)
        if prec == 0:
            scratch = torch.empty(_C.eval_topk_scratch_bytes(bs, I, k), dtype=torch.uint8, device=dev)
        else:
            scratch = torch.empty(_C.eval_topk_tc_scratch_bytes(bs, I, kc), dtype=torch.uint8, device=dev)
            Vq = _C.pack_rows(Vfull[:, :lay.d], lay.d, prec)
        top_s = torch.empty((bs, k), dtype=torch.float32, device=dev)
        top_i = torch.empty((bs, k), dtype=torch.int32, device=dev)
        cand_s = torch.empty((bs, kc), dtype=torch.float32, device=dev) if kc > k else None
        cand_i = torch.empty((bs, kc), dtype=torch.int32, device=dev) if kc > k else None
        evaluator._prepare(dev)
        for s0 in range(0, n_loc, bs):
            n = min(bs, n_loc - s0)
            rows_l = torch.arange(s0, s0 + n, dtype=torch.int64, device=dev)      # local user rows
            gids = rows_l * G + r                                                   # their global ids (exclusion / label rows)
            if prec == 0:
                _C.eval_topk(t, gids, k, top_s[:n], top_i[:n], scratch, exclude.indptr, exclude.indices, status=self.status,
                             u_rows=rows_l, n_users_global=self.spec.n_users)
            else:
                Uq = _C.pack_rows(U2d[:, :lay.d], lay.d, prec, row_idx=rows_l)
                cs, ci = (cand_s[:n], cand_i[:n]) if kc > k else (top_s[:n], top_i[:n])
                _C.eval_topk_tc(Uq, Vq, prec, gids, self.spec.n_users, kc, cs, ci, scratch, Ub=Ub, Ib=Ibfull, Gb=Gb,
                                excl_indptr=exclude.indptr, excl_indices=exclude.indices, status=self.status, u_rows=rows_l)
                if kc > k:
                    _C.rescore_topk(t, rows_l, ci, k, top_s[:n], top_i[:n], status=self.status, cand_scores=cs)
            evaluator.eval_batch_topk(gids, top_i[:n].contiguous(), labels)
        self._reduce_metric_sums(evaluator)
        return evaluator.get_results()


    def _map_peers(self, tensors: Dict[str, torch.Tensor], extra: Dict[str, int]):
        """Collective: export `tensors` (name -> device tensor) to the peers of this node and map theirs.  Returns per rank q
        a dict name -> address in THIS process, plus the peers' `extra` integers."""
        G, r = self.spec.world, self.spec.rank
        mine = dict(extra)
        if G > 1:
            import socket
            mine['host'] = socket.gethostname()
            try:
                mine['exports'] = {n: _C.peer_export(t) for n, t in tensors.items()}
            except _C.HskError as ex:
                mine['error'] = str(ex)
            every = [None] * G
            dist.all_gather_object(every, mine, group=self.group)
            errs = [f"rank {q}: {e['error']}" for q, e in enumerate(every) if 'error' in e]
            if errs or len({e['host'] for e in every}) != 1:
                raise _C.HskError('peer mapping is not available (' + ('; '.join(errs) or 'the ranks are not on one node') + ')')
        else:
            every = [mine]
        out, failure = [], None
        try:
            for q in range(G):
                d = {k: v for k, v in every[q].items() if k not in ('exports', 'host')}
                for n, t in tensors.items():
                    if q == r:
                        d[n] = t.data_ptr()
                    else:
                        handle, off = every[q]['exports'][n]
                        if (q, handle) not in self._ipc:
                            self._ipc[(q, handle)] = _C.peer_open(handle, self.device)
                        d[n] = self._ipc[(q, handle)] + off
                out.append(d)
        except _C.HskError as ex:
            failure = str(ex)
        if G > 1:
            ok = torch.tensor([0 if failure else 1], dtype=torch.int32, device=self.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if int(ok.item()) == 0:
                raise _C.HskError('peer mapping is not available (' + (failure or 'failed on another rank') + ')')
        elif failure:
            raise _C.HskError(failure)
        return out

    def evaluate_streamed(self, labels_csr, exclude_csr, evaluator, batch_size: int = 18944, precision: str = 'bf16',
                          rescore: bool = True, max_users: Optional[int] = None):
        """Item-SHARDED tables, user-parallel scoring (one NVLink / NVSwitch node, tensor-core precisions): the item shards stay
        where they are; every rank evaluates ITS users against ALL items with one kernel per batch that reads the other ranks'
        packed item tables straight from their HBM (TMA loads over CUDA IPC mappings) and re-scores its candidates in fp32 from
        the owners' rows the same way.  No replica (unlike `evaluate_replicated`), no per-shard candidate lists, no merge, no
        per-round collective (unlike `evaluate`); results are exactly the single-GPU results.
        Cost, measured: peer rows are NOT cached in the reader's L2, so each of the 74 CTA pairs of a launch pulls the remote
        shards over the link itself — ~37 GB x (G - 1) / G per 18 944-user batch at cfg5 against ~640 GB/s — 37 ms per batch on
        2 GPUs where the replicated mode needs 11.  Use it for catalogues whose packed item table does not fit one GPU (the only
        case that needs item-sharded STORAGE); otherwise `evaluate_replicated` (1.5 GB at cfg5) is 3x faster and `evaluate` keeps
        memory per GPU at 1 / G.  `max_users`: bound on the LOCAL users evaluated (bench samples)."""
        from hassaku_b200.eval.eval import DeviceCSR
        if precision not in ('tf32', 'bf16'):
            raise ValueError("evaluate_streamed scores on the tensor cores: precision 'tf32' or 'bf16' (fp32-exact: evaluate / "
                             "evaluate_replicated)")
        prec = _C.PRECISIONS[precision]
        G, r, lay, dev = self.spec.world, self.spec.rank, self.layout, self.device
        k = max(evaluator.K_VALUES)
        labels = labels_csr if isinstance(labels_csr, DeviceCSR) else self._csr_cache(labels_csr)
        exclude = exclude_csr if isinstance(exclude_csr, DeviceCSR) else self._csr_cache(exclude_csr)
        Uw, Vw, Ub, Ib, Gb = lay.views(self.arena)
        # this rank's shard, packed once per sweep into a buffer that lives as long as the model (one IPC mapping per peer)
        cache = self.__dict__.setdefault('_vq_cache', {})
        Vq = cache[prec] = _C.pack_rows(Vw.detach(), lay.d, prec, out=cache.get(prec))
        peers = self._map_peers({'Vq': Vq, 'arena': self.arena}, {'rows': lay.n_items, 'off_V': lay.off_V, 'off_Ib': lay.off_Ib})
        shards = _C.ItemShards([p['rows'] for p in peers], Vq=[p['Vq'] for p in peers],
                               V=[p['arena'] + 4 * p['off_V'] for p in peers],
                               Ib=[p['arena'] + 4 * p['off_Ib'] for p in peers] if Ib is not None else None)
        torch.cuda.synchronize(dev)
        if G > 1:
            dist.barrier(group=self.group)                        # every rank's packed shard is complete before anyone streams it
        n_loc = lay.n_users if max_users is None else min(lay.n_users, max_users)
        bs = max(1, min(batch_size, n_loc))
        kc = min(128, k + self.RESCORE_MARGIN, self.spec.n_items) if rescore else k
        U2d = self._table2d(self.arena, 'U')
        t_user = _C.make_tables(U2d[:, :lay.d], self._table2d(self.arena, 'V')[:, :lay.d], Ub, Ib, Gb, lay.d)
        scratch = torch.empty(_C.eval_topk_tc_shards_scratch_bytes(bs, shards, kc), dtype=torch.uint8, device=dev)
        top_s = torch.empty((bs, k), dtype=torch.float32, device=dev)
        top_i = torch.empty((bs, k), dtype=torch.int32, device=dev)
        cand_s = torch.empty((bs, kc), dtype=torch.float32, device=dev) if kc > k else None
        cand_i = torch.empty((bs, kc), dtype=torch.int32, device=dev) if kc > k else None
        evaluator._prepare(dev)
        for s0 in range(0, n_loc, bs):
            n = min(bs, n_loc - s0)
            rows_l = torch.arange(s0, s0 + n, dtype=torch.int64, device=dev)      # local user rows
            gids = rows_l * G + r                                                   # their global ids (exclusion / label rows)
            Uq = _C.pack_rows(U2d[:, :lay.d], lay.d, prec, row_idx=rows_l)
            cs, ci = (cand_s[:n], cand_i[:n]) if kc > k else (top_s[:n], top_i[:n])
            _C.eval_topk_tc_shards(Uq, shards, prec, gids, self.spec.n_users, kc, cs, ci, scratch, Ub=Ub, Gb=Gb,
                                   excl_indptr=exclude.indptr, excl_indices=exclude.indices, status=self.status, u_rows=rows_l)
            if kc > k:
                _C.rescore_topk_shards(t_user, shards, rows_l, ci, k, top_s[:n], top_i[:n], status=self.status, cand_scores=cs)
            evaluator.eval_batch_topk(gids, top_i[:n].contiguous(), labels)
        self._reduce_metric_sums(evaluator)
        torch.cuda.synchronize(dev)
        if G > 1:
            dist.barrier(group=self.group)                        # nobody still reads this rank's packed shard when it is freed
        return evaluator.get_results()


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def partition_batch_by_user_owner(u_idxs: torch.Tensor, i_idxs: torch.Tensor, world: int, rank: int):
    """The rows of a GLOBAL batch this rank processes (sample -> owner of its user, SURVEY §8e)."""
    sel = (u_idxs % world) == rank
    return u_idxs[sel].contiguous(), i_idxs[sel].contiguous()
