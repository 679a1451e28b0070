"""Phase times of one item-sharded evaluation round (cfg5 shape), without stream overlap: where a round's time goes.
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 scripts/eval_phases.py [--users-per-round 18944]
"""
import argparse
import math
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hassaku_b200 import _C  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--users-per-round', type=int, default=18944)
    ap.add_argument('--items', type=int, default=1_000_000)
    ap.add_argument('--dim', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=6)
    a = ap.parse_args()
    rank, G = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', 0)))
    torch.cuda.set_device(dev)
    if G > 1:
        dist.init_process_group('nccl', device_id=dev)
    d, k, kc = a.dim, 100, 128
    nl = len(range(rank, a.items, G))
    Be, bs = a.users_per_round, a.users_per_round // G
    g = torch.Generator(device=dev); g.manual_seed(rank)
    V = torch.randn((nl, d), device=dev, generator=g) / math.sqrt(d)
    Ib = torch.randn(nl, device=dev, generator=g) * 0.05
    rows = torch.randn((bs, d), device=dev, generator=g) / math.sqrt(d)
    all_rows = torch.empty((Be, d), device=dev)
    P = _C.PRECISIONS['bf16']
    Vq = _C.pack_rows(V, d, P)
    users = torch.arange(Be, device=dev)
    scratch = torch.empty(_C.eval_topk_tc_scratch_bytes(Be, nl, kc), dtype=torch.uint8, device=dev)
    cs, ci = torch.empty((Be, kc), device=dev), torch.empty((Be, kc), dtype=torch.int32, device=dev)
    rs, ri = torch.empty((G, bs, kc), device=dev), torch.empty((G, bs, kc), dtype=torch.int32, device=dev)
    mcs, mci = torch.empty((bs, kc), device=dev), torch.empty((bs, kc), dtype=torch.int32, device=dev)
    all_mci = torch.empty((Be, kc), dtype=torch.int32, device=dev)
    sc, rsc = torch.empty((Be, kc), device=dev), torch.empty((G, bs, kc), device=dev)
    ms, mi = torch.empty((bs, k), device=dev), torch.empty((bs, k), dtype=torch.int32, device=dev)
    t = _C.make_tables(all_rows, V, None, Ib, None, d)

    def coll(fn, *x):
        if G > 1:
            fn(*x)
    phases = {}

    def timed(name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        phases.setdefault(name, []).append((e0, e1))

    for r in range(a.rounds):
        timed('all_gather rows', lambda: dist.all_gather_into_tensor(all_rows, rows) if G > 1 else all_rows.copy_(rows))
        box = {}
        timed('pack_rows', lambda: box.__setitem__('Uq', _C.pack_rows(all_rows, d, P)))
        timed('eval_topk_tc', lambda: _C.eval_topk_tc(box['Uq'], Vq, P, users, Be, kc, cs, ci, scratch, Ib=Ib, id_offset=rank, id_stride=G))
        timed('a2a lists x2', lambda: (coll(dist.all_to_all_single, rs, cs.view(G, bs, kc)), coll(dist.all_to_all_single, ri, ci.view(G, bs, kc))))
        if G == 1:
            rs.copy_(cs.view(G, bs, kc)); ri.copy_(ci.view(G, bs, kc))
        timed('topk_merge kc', lambda: _C.topk_merge(rs, ri, mcs, mci))
        timed('all_gather ids', lambda: dist.all_gather_into_tensor(all_mci, mci) if G > 1 else all_mci.copy_(mci))
        timed('rescore_scores', lambda: _C.rescore_scores(t, users, all_mci, sc, id_offset=rank, id_stride=G))
        timed('a2a scores', lambda: coll(dist.all_to_all_single, rsc, sc.view(G, bs, kc)))
        if G == 1:
            rsc.copy_(sc.view(G, bs, kc))
        timed('topk_combine', lambda: _C.topk_combine(rsc, mci, k, ms, mi, cand_scores=mcs))
    torch.cuda.synchronize()
    if rank == 0:
        tot = 0.0
        for name, evs in phases.items():
            v = sorted(x.elapsed_time(y) for x, y in evs[1:])
            med = v[len(v) // 2]
            tot += med
            print(f'{name:18s} {med * 1e3:9.1f} us')
        print(f'{"sum":18s} {tot * 1e3:9.1f} us   (G = {G}, {Be} users / round, {nl} local items)')
    if G > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
