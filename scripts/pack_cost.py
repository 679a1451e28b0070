"""What a trial pack buys: M BPR-MF trials trained as one pack (PackedMFTrainStep: one fused-step launch, one row-stamp
launch and one AdamW launch per step for all M) against the same M trials trained one after the other through Trainer's
step path (FusedMFTrainStep + DenseAdam, one model at a time), at the ML-1M shape (6 040 x 3 706).

Grid: d in {64, 402} x (B, neg_train) in {(64, 4) the reference default, (1024, 4), (8192, 50)} x M in {1, 4, 16, 64}.
The two arms alternate window by window; a window is K steps of every trial (packed: K pack steps; single: K steps of
trial 0, then K of trial 1, ...), timed with CUDA events.  Steps run back to back as in training (no L2 flush).  Batches:
uniform random users and items, pre-generated on the device.  An epoch is 1 000 000 interactions (the ML-1M shape of
data/synthetic.py) / B steps; trial-epochs/s = M / (steps per epoch x time of one step of all M trials), i.e. whole epochs
extrapolated from the timed windows.  Writes JSON with the GPU name and power limit (nvidia-smi query in the same run).
    python scripts/pack_cost.py [--k 20] [--rounds 5] [--out profiles/pack_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U, I, N_INTER = 6040, 3706, 1_000_000
LR, WD = 3e-4, 4e-5


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def _models(M, d, seed0):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    return [SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=seed0 + j) for j in range(M)]


def measure(d, B, N, M, k, rounds):
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    from hassaku_b200.train.trial_pack import PackedMFTrainStep
    loss = RecBayesianPersonalizedRankingLoss()
    lrs = [LR * (1 + 0.1 * j) for j in range(M)]
    wds = [WD if j % 2 else 0.0 for j in range(M)]
    pack = PackedMFTrainStep(_models(M, d, 100), loss, lrs, wds)
    singles = []
    for j, mdl in enumerate(_models(M, d, 100)):
        singles.append(FusedMFTrainStep(mdl, loss, DenseAdam(mdl, lr=lrs[j], weight_decay=wds[j])))
    gen = torch.Generator(device='cuda')
    gen.manual_seed(5)
    batches = [(torch.randint(0, U, (B,), device='cuda', generator=gen),
                torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)) for _ in range(8)]
    times = {'packed': [], 'single': []}
    for r in range(rounds + 1):                       # round 0 warms up both arms
        for arm in ('packed', 'single'):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if arm == 'packed':
                pack.prepare(k)
            a.record()
            if arm == 'packed':
                for s in range(k):
                    pack.step(*batches[s % len(batches)])
            else:
                for st in singles:
                    for s in range(k):
                        st(*batches[s % len(batches)])
            b.record()
            torch.cuda.synchronize()
            if r > 0:
                times[arm].append(a.elapsed_time(b) / k)     # ms per step of all M trials
    pack.pop_loss_sums()
    for st in singles:
        st.pop_loss_sum()
    steps_per_epoch = -(-N_INTER // B)
    out = {'d': d, 'B': B, 'neg_train': N, 'M': M, 'steps_per_epoch': steps_per_epoch,
           'pack_bytes_adamw_per_step': 28 * pack.stride * M}
    for arm, ts in times.items():
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        out[arm] = {'ms_per_step_all_trials_median': med, 'min': ts[0], 'max': ts[-1],
                    'trial_epochs_per_s': M / (steps_per_epoch * med * 1e-3)}
    out['ratio_packed_over_single'] = out['packed']['trial_epochs_per_s'] / out['single']['trial_epochs_per_s']
    del pack, singles
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--k', type=int, default=20, help='steps of every trial per timed window')
    ap.add_argument('--rounds', type=int, default=5, help='timed windows per arm (alternating)')
    ap.add_argument('--dims', default='64,402')
    ap.add_argument('--shapes', default='64x4,1024x4,8192x50')
    ap.add_argument('--packs', default='1,4,16,64')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'pack_cost.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('pack_cost.py measures on a CUDA device; none is available')
    res = {'gpu': gpu_info(), 'shape': {'n_users': U, 'n_items': I, 'epoch_interactions': N_INTER, 'loss': 'bpr',
                                         'item_bias': True, 'optimizer': 'adamw'},
           'k': args.k, 'rounds': args.rounds, 'l2': 'no flush: consecutive steps as in training', 'results': []}
    for d in [int(x) for x in args.dims.split(',')]:
        for shp in args.shapes.split(','):
            B, N = [int(x) for x in shp.split('x')]
            for M in [int(x) for x in args.packs.split(',')]:
                r = measure(d, B, N, M, args.k, args.rounds)
                print(json.dumps(r), flush=True)
                res['results'].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
