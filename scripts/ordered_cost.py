"""Cost of the sharded step's ORDERED exchange (ShardedMF.step(exchange='ordered_graph'), the deterministic multi-GPU
step) on one GPU, at the cfg4 and cfg2 shapes of bench.py.  Four arms from one initial model, alternated step by step on
the same batches, CUDA events per step:
  single_default   FusedMFTrainStep + DenseAdam (hsk_mf_train_fused, the single-GPU default step)
  single_det       the same under torch.use_deterministic_algorithms(True) (hsk_mf_train_fused_det)
  sparse_graph     ShardedMF(world=1), exchange='sparse_graph' (the non-deterministic sharded step)
  ordered_graph    ShardedMF(world=1), exchange='ordered_graph', under the switch
At world 1 the ordered step is the single-GPU deterministic step bit for bit; the script checks that on the final
parameters.  Then one profiled run (torch.profiler, CUDA activities) of eager ordered steps splits the ordered step's
kernel time by phase.  The L2 is flushed before every timed step at cfg2 (tables and optimizer state fit the 126 MB L2),
as bench.py does, not in the profiled run.  Batches: uniform random users and items.  Writes JSON (GPU name and power limit included).
    python scripts/ordered_cost.py [--warmup 20] [--steps 200] [--out profiles/ordered_cost.json]
"""
import argparse
import collections
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

DIMS = {'ml1m': (6040, 3706), 'ml10m': (69_878, 10_677), 'lfm2b': (2_000_000, 1_000_000)}   # data/synthetic.py
ARMS = ('single_default', 'single_det', 'sparse_graph', 'ordered_graph')
# kernel name fragment -> phase of the ordered step (first match wins)
PHASES = (('route_', 'routing'), ('shard_pack', 'pack'), ('det_forward', 'det forward'), ('sort_', 'sorts'),
          ('scan_', 'sorts'), ('det_chunk', 'chunk/combine'), ('det_combine', 'chunk/combine'), ('gb_', 'chunk/combine'),
          ('det_loss_sum', 'loss sum'), ('shard_unpack_ordered', 'unpack'), ('adamw', 'AdamW'), ('mark_rows', 'routing'),
          ('shard_local_index', 'routing'))


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def phase_of(name):
    for frag, ph in PHASES:
        if frag in name:
            return ph
    return 'copies / memsets / other'


def measure(wname, warmup, steps, flush, prof_steps):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.sharded import ShardedMF
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import RecommenderSystemLossesEnum
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    name, d, B, N, loss, lr, wd = bench.WORKLOADS[wname]
    U, I = DIMS[name]

    class _DS:
        n_items = I

    model = SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=64)
    sd0 = {k: v.detach() for k, v in model.state_dict().items()}
    model_det = SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=64)
    build = lambda m: FusedMFTrainStep(m, RecommenderSystemLossesEnum[loss].value.build_from_conf(   # noqa: E731
        {'train_neg_strategy': 'uniform', 'neg_train': N}, _DS()), DenseAdam(m, lr=lr, weight_decay=wd))
    single, single_det = build(model), build(model_det)
    kind, shift = single.rec_loss.loss_kind, single.shift
    shards = {}
    for arm in ('sparse_graph', 'ordered_graph'):
        shards[arm] = ShardedMF(U, I, d, use_item_bias=True, world=1, rank=0, device='cuda')
        shards[arm].load_full_state_dict(sd0)
    del sd0
    gen = torch.Generator(device='cuda')
    gen.manual_seed(5)
    batches = [(torch.randint(0, U, (B,), device='cuda', generator=gen),
                torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)) for _ in range(16)]

    def run(arm, u, i):
        if arm == 'single_default':
            single(u, i)
        elif arm == 'single_det':
            single_det(u, i)
        else:
            shards[arm].step(u, i, B, kind, shift, lr, wd, exchange=arm)

    small = wname != 'cfg4'
    times = {a: [] for a in ARMS}
    for k in range(len(ARMS) * (warmup + steps)):
        arm = ARMS[k % len(ARMS)]
        u, i = batches[(k // len(ARMS)) % len(batches)]
        if small:
            flush.zero_()
        torch.use_deterministic_algorithms(arm in ('single_det', 'ordered_graph'))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run(arm, u, i)
        b.record()
        torch.use_deterministic_algorithms(False)
        torch.cuda.synchronize()
        if k >= len(ARMS) * warmup:
            times[arm].append(a.elapsed_time(b))
    # every arm took the same steps on the same batches: the ordered step at world 1 is the single-GPU deterministic step
    got = shards['ordered_graph'].full_state_dict(to_cpu=False)
    same = all(torch.equal(got[n].view(torch.int32), p.detach().view(torch.int32)) for n, p in model_det.state_dict().items())
    losses = {'single_det': single_det.pop_loss_sum(), 'ordered_graph': shards['ordered_graph'].pop_loss(),
              'single_default': single.pop_loss_sum(), 'sparse_graph': shards['sparse_graph'].pop_loss()}
    out = {'workload': wname, 'shape': {'n_users': U, 'n_items': I, 'd': d, 'B': B, 'N': N, 'loss': loss},
           'l2': 'flushed before every timed step' if small else 'inputs larger than L2, no flush',
           'ordered_equals_single_det_bitwise': bool(same and losses['single_det'] == losses['ordered_graph']),
           'loss_sums': losses}
    for arm, ts in times.items():
        ts = sorted(ts)
        out[arm] = {'median_ms': ts[len(ts) // 2], 'p10_ms': ts[len(ts) // 10], 'p90_ms': ts[9 * len(ts) // 10]}
    for arm in ARMS[1:]:
        out[f'{arm}_over_single_default'] = out[arm]['median_ms'] / out['single_default']['median_ms']
    out['ordered_graph_over_sparse_graph'] = out['ordered_graph']['median_ms'] / out['sparse_graph']['median_ms']
    out['ordered_graph_over_single_det'] = out['ordered_graph']['median_ms'] / out['single_det']['median_ms']
    for sm in shards.values():
        sm.close()
    # per-phase kernel time of the eager ordered step (a separate profiled run)
    eager = shards['ordered_graph']
    torch.use_deterministic_algorithms(True)
    for k in range(3):
        eager.step(*batches[k], B, kind, shift, lr, wd, exchange='ordered')
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(prof_steps):
            eager.step(*batches[k % len(batches)], B, kind, shift, lr, wd, exchange='ordered')
        torch.cuda.synchronize()
    torch.use_deterministic_algorithms(False)
    per = collections.defaultdict(float)
    for ev in prof.key_averages():
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        if us > 0:
            per[phase_of(ev.key)] += us / 1000.0 / prof_steps
    out['phase_note'] = 'eager ordered steps back to back, no L2 flush between them'
    out['ordered_eager_kernel_ms_per_step_by_phase'] = {k: round(v, 4) for k, v in sorted(per.items(), key=lambda x: -x[1])}
    out['ordered_eager_kernel_ms_per_step_total'] = round(sum(per.values()), 4)
    del model, model_det, single, single_det, shards, eager
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--profile-steps', type=int, default=20)
    ap.add_argument('--workloads', default='cfg4,cfg2')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'ordered_cost.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('ordered_cost.py measures on a CUDA device; none is available')
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')   # > 126 MB L2
    res = {'gpu': gpu_info(), 'warmup': args.warmup, 'steps': args.steps, 'world': 1,
           'note': 'N > 1 (torchrun against the peer / sparse exchanges) not measured',
           'results': [measure(w, args.warmup, args.steps, flush, args.profile_steps) for w in args.workloads.split(',')]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
