"""What packed validation buys: the validation of M MF trials of one trial pack as one packed sweep (evaluate_mf_pack:
per chunk of users one hsk_eval_topk_pack and one hsk_rank_metrics_pack launch for all M) against M sequential
evaluate_recommender_algorithm calls (PackedTrainer.val per trial, what the trainer ran before), on the validation split of
the ML-1M-shaped synthetic data (data/synthetic.py: 6 040 users x 3 706 items, 1 000 000 interactions).

Grid: d in {64, 402} x eval loader batch in {64, 1024} x M in {1, 4, 16, 64}.  The two arms alternate; each call ends in
the sweep's host sync and is timed with a host clock.  Round 0 warms up both arms.  The packed arm's FP32 rate is
2 * U * I * d * M FLOP (the scoring contraction, no exclusions skipped) over its time.

Epoch split: for the pack_cost.py shapes (d in {64, 402} x (B, neg_train) in {(64, 4), (1024, 4), (8192, 50)}) at M = 64,
one PackedTrainer.fit epoch = the packed training epoch (PackedMFTrainStep steps of the 64 trials, timed with CUDA events
in this run and extrapolated to 1 000 000 / B steps) + one validation at eval batch 64: before = sequential, after =
packed.  Writes JSON with the GPU name, power limit and max SM clock (nvidia-smi query in the same run).
    python scripts/eval_pack_cost.py [--rounds 3] [--out profiles/eval_pack_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U, I, N_INTER = 6040, 3706, 1_000_000


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


class _EvalLoader:
    def __init__(self, dataset, batch_size):
        self.dataset, self.batch_size = dataset, batch_size


def _pack_models(M, d, seed0=100):
    """M trials bound to the rows of one [M, stride] allocation, as PackedMFTrainStep binds them."""
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    models = [SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=seed0 + j, std=(d ** -0.5, 0.05))
              for j in range(M)]
    p = torch.empty((M, models[0].layout.n_total), dtype=torch.float32, device='cuda')
    for j, m in enumerate(models):
        p[j].copy_(m.arena.detach())
        m._set_arena(p[j])
    return models, p


def measure_val(ds, d, bs, M, rounds):
    from hassaku_b200.eval.eval import FullEvaluator, evaluate_mf_pack, evaluate_recommender_algorithm, pack_chunk_users
    models, p = _pack_models(M, d)
    loader = _EvalLoader(ds, bs)
    mk = lambda: FullEvaluator(aggr_by_group=True, n_groups=ds.n_user_groups, user_to_user_group=ds.user_to_user_group)
    times = {'packed': [], 'sequential': []}
    agree = True
    for r in range(rounds + 1):
        for arm in ('packed', 'sequential'):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if arm == 'packed':
                got = evaluate_mf_pack(models, loader, [mk() for _ in range(M)], 'cuda')
            else:
                want = [evaluate_recommender_algorithm(m, loader, mk(), 'cuda') for m in models]
            dt = time.perf_counter() - t0
            if r > 0:
                times[arm].append(dt)
        agree = agree and all(g['ndcg@10'] == w['ndcg@10'] and g['recall@100'] == w['recall@100'] for g, w in zip(got, want))
    out = {'d': d, 'eval_batch': bs, 'M': M, 'chunk_users': pack_chunk_users(bs, U, I, 100, M),
           'metrics_equal': agree}
    for arm, ts in times.items():
        ts = sorted(ts)
        out[arm] = {'s_median': ts[len(ts) // 2], 'min': ts[0], 'max': ts[-1]}
    flop = 2.0 * ds.n_users * I * d * M
    out['packed_fp32_tflops'] = flop / out['packed']['s_median'] / 1e12
    out['sequential_fp32_tflops'] = flop / out['sequential']['s_median'] / 1e12
    out['speedup_packed'] = out['sequential']['s_median'] / out['packed']['s_median']
    del models, p
    torch.cuda.empty_cache()
    return out


def measure_train_epoch(d, B, N, M, k):
    """Seconds of one packed training epoch (1 000 000 / B steps of all M trials), from k timed steps after k warm-up."""
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trial_pack import PackedMFTrainStep
    models = [SGDMatrixFactorization.on_device(U, I, d, use_item_bias=True, seed=100 + j) for j in range(M)]
    pack = PackedMFTrainStep(models, RecBayesianPersonalizedRankingLoss(), [3e-4] * M, [4e-5] * M)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(5)
    batches = [(torch.randint(0, U, (B,), device='cuda', generator=gen),
                torch.randint(0, I, (B, N + 1), device='cuda', generator=gen)) for _ in range(8)]
    pack.prepare(2 * k)
    for s in range(k):
        pack.step(*batches[s % len(batches)])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for s in range(k):
        pack.step(*batches[s % len(batches)])
    b.record()
    torch.cuda.synchronize()
    pack.pop_loss_sums()
    ms = a.elapsed_time(b) / k
    del pack, models
    torch.cuda.empty_cache()
    return ms * 1e-3 * -(-N_INTER // B)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3, help='timed calls per arm (alternating)')
    ap.add_argument('--dims', default='64,402')
    ap.add_argument('--batches', default='64,1024')
    ap.add_argument('--packs', default='1,4,16,64')
    ap.add_argument('--train-shapes', default='64x4,1024x4,8192x50')
    ap.add_argument('--train-k', type=int, default=40, help='timed packed training steps per shape')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'eval_pack_cost.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('eval_pack_cost.py measures on a CUDA device; none is available')
    from hassaku_b200.data.dataset import FullEvalDataset
    from hassaku_b200.data.synthetic import make_interactions
    data = make_interactions(U, I, N_INTER, seed=0, n_user_groups=2)
    ds = FullEvalDataset.from_interactions(data.val, data.train, 'val', data.user_group, 2)
    res = {'gpu': gpu_info(), 'shape': {'n_users': ds.n_users, 'n_items': ds.n_items, 'interactions': N_INTER,
                                        'split': 'val', 'user_groups': 2, 'k_values': [5, 10, 50, 100]},
           'rounds': args.rounds, 'timing': 'host clock around calls that end in the sweep\'s host sync',
           'validation': [], 'epoch_split_M64': []}
    val = {}
    for d in [int(x) for x in args.dims.split(',')]:
        for bs in [int(x) for x in args.batches.split(',')]:
            for M in [int(x) for x in args.packs.split(',')]:
                r = measure_val(ds, d, bs, M, args.rounds)
                val[(d, bs, M)] = r
                print(json.dumps(r), flush=True)
                res['validation'].append(r)
    for d in [int(x) for x in args.dims.split(',')]:
        v = val.get((d, 64, 64))
        if v is None:
            continue
        for shp in args.train_shapes.split(','):
            B, N = [int(x) for x in shp.split('x')]
            train_s = measure_train_epoch(d, B, N, 64, args.train_k)
            before, after = v['sequential']['s_median'], v['packed']['s_median']
            r = {'d': d, 'B': B, 'neg_train': N, 'M': 64, 'eval_batch': 64, 'train_epoch_s': train_s,
                 'val_before_s': before, 'val_after_s': after,
                 'val_share_before': before / (train_s + before), 'val_share_after': after / (train_s + after),
                 'epoch_speedup': (train_s + before) / (train_s + after)}
            print(json.dumps(r), flush=True)
            res['epoch_split_M64'].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
