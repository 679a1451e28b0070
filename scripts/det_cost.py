"""Cost of the deterministic mode: the default fused training step (hsk_mf_train_fused + AdamW) against the same step under
torch.use_deterministic_algorithms(True) (hsk_mf_train_fused_det + AdamW), at the cfg2 / cfg3 / cfg4 shapes of bench.py.
The two arms alternate step by step from one model; CUDA events per step; the L2 is flushed before every timed step at
cfg2 / cfg3 (tables and optimizer state fit the 126 MB L2) as bench.py does.  Batches: uniform random users and items
(the step's cost depends on the shape, not on the sampler).  Writes JSON (GPU name and power limit included).
    python scripts/det_cost.py [--warmup 20] [--steps 200] [--out profiles/det_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

DIMS = {'ml1m': (6040, 3706), 'ml10m': (69_878, 10_677), 'lfm2b': (2_000_000, 1_000_000)}   # data/synthetic.py


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def measure(wname, warmup, steps, flush):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import RecommenderSystemLossesEnum
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    name, d, B, N, loss, lr, wd = bench.WORKLOADS[wname]
    U, I = DIMS[name]

    class _DS:
        n_items = I

    model = SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=64)
    opt = DenseAdam(model, lr=lr, weight_decay=wd)
    step = FusedMFTrainStep(model, RecommenderSystemLossesEnum[loss].value.build_from_conf(
        {'train_neg_strategy': 'uniform', 'neg_train': N}, _DS()), opt)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(5)
    batches = [(torch.randint(0, U, (B,), device='cuda', generator=gen),
                torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)) for _ in range(16)]
    big = wname == 'cfg4'
    times = {'default': [], 'deterministic': []}
    for k in range(2 * (warmup + steps)):
        arm = 'deterministic' if k % 2 else 'default'
        u, i = batches[(k // 2) % len(batches)]
        if not big:
            flush.zero_()
        torch.use_deterministic_algorithms(arm == 'deterministic')
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(u, i)
        b.record()
        torch.use_deterministic_algorithms(False)
        torch.cuda.synchronize()
        if k >= 2 * warmup:
            times[arm].append(a.elapsed_time(b))
    step.pop_loss_sum()
    out = {'workload': wname, 'shape': {'n_users': U, 'n_items': I, 'd': d, 'B': B, 'N': N, 'loss': loss},
           'l2': 'inputs larger than L2, no flush' if big else 'flushed before every timed step'}
    for arm, ts in times.items():
        ts = sorted(ts)
        out[arm] = {'median_ms': ts[len(ts) // 2], 'p10_ms': ts[len(ts) // 10], 'p90_ms': ts[9 * len(ts) // 10]}
    out['ratio_median'] = out['deterministic']['median_ms'] / out['default']['median_ms']
    del model, opt, step
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--workloads', default='cfg2,cfg3,cfg4')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'det_cost.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('det_cost.py measures on a CUDA device; none is available')
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')   # > 126 MB L2
    res = {'gpu': gpu_info(), 'warmup': args.warmup, 'steps': args.steps,
           'results': [measure(w, args.warmup, args.steps, flush) for w in args.workloads.split(',')]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
