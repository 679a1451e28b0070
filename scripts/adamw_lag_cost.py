"""Cost of the cfg4 training step against the m / v write-back period of DenseAdam (state_lag, hsk_adamw_dense_rows_lag).

    python scripts/adamw_lag_cost.py [--lags 1,2,4,8,16] [--rounds 3] [--steps 200] [--hash-steps 30]

One process, the bench's cfg4 workload (2 M users x 1 M items x d 128 + item bias, B 8192, N 50, BPR, AdamW lr 3e-4
wd 4e-5; bench.make_device_batches on make_device_interactions, 16 distinct batches):
  * bitwise check: under torch.use_deterministic_algorithms(True), per lag a fresh model (seed 64) takes --hash-steps
    FusedMFTrainStep steps; p is hashed after them, then m and v (DenseAdam.m / .v sync every row first).  Equal hashes
    across lags: the lagged moments change nothing at full size;
  * timing: one model + optimizer per lag, all resident; the arms alternate --rounds times, each round --warmup steps
    then CUDA events around --steps steps (whole step), then 50 steps with events between the fused kernel, the marking
    launch and the AdamW launch (the bench's per-kernel split).  The 6.2 GB per arm is far beyond the 126 MB L2;
  * modelled AdamW bytes per step from the rows the batches stamp: untouched parameters 16 + 8 / K bytes (24 at K = 1),
    stamped ones 32, the bias vector 32, the base bytes 2 per row for K > 1.
Writes --out (JSON) with the card's name, power limit and clocks read in the same run."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U, I, D, B, N = 2_000_000, 1_000_000, 128, 8192, 50
LR, WD = 3e-4, 4e-5
N_DISTINCT = 16


def gpu_info():
    q = 'name,power.limit,clocks.max.sm,clocks.sm,clocks.mem'
    try:
        r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], capture_output=True, text=True,
                           timeout=60)
        return dict(zip(q.split(','), [x.strip() for x in r.stdout.splitlines()[0].split(',')]))
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return {'error': str(e)}


def _arm(lag, dev):
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.train.optim import DenseAdam
    from hassaku_b200.train.rec_losses import RecBayesianPersonalizedRankingLoss
    from hassaku_b200.train.trainer_step import FusedMFTrainStep
    model = SGDMatrixFactorization.on_device(U, I, D, use_item_bias=True, device=dev, seed=64)
    opt = DenseAdam(model, lr=LR, weight_decay=WD, decoupled=True, state_lag=lag)
    return model, opt, FusedMFTrainStep(model, RecBayesianPersonalizedRankingLoss(), opt)


def _sha(t):
    import torch
    h = hashlib.sha256()
    for c in t.detach().view(torch.int32).split(1 << 26):
        h.update(c.cpu().numpy().tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--lags', default='1,2,4,8,16')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--hash-steps', type=int, default=30)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'adamw_lag_cost.json'))
    args = ap.parse_args()
    import torch
    from bench import make_device_batches
    from hassaku_b200 import _C
    from hassaku_b200.data.synthetic import SHAPES, make_device_interactions
    lags = [int(x) for x in args.lags.split(',')]
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    info = {'gpu_before': gpu_info()}
    _, _, n_inter = SHAPES['lfm2b']
    data = make_device_interactions(U, I, n_inter, dev, 1, 0, seed=0)
    us, its = make_device_batches(data, B, N, N_DISTINCT)
    del data

    # ---- touched rows per step (the stamps of the batches) and modelled bytes ----
    tu = [int(torch.unique(u).numel()) for u in us]
    ti = [int(torch.unique(i).numel()) for i in its]
    touched_users, touched_items = statistics.mean(tu), statistics.mean(ti)
    P = U * D + I * D
    touched_p = (touched_users + touched_items) * D

    def model_bytes(K):
        untouched = (P - touched_p) * ((16 + 8 / K) if K > 1 else 24)
        return untouched + touched_p * 32 + I * 32 + (2 * (U + I) if K > 1 else 0)

    # ---- bitwise: p after hash_steps deterministic steps, m / v after a sync ----
    hashes = {}
    prev = torch.are_deterministic_algorithms_enabled()
    for K in lags:
        model, opt, step = _arm(K, dev)
        torch.use_deterministic_algorithms(True)
        for s in range(args.hash_steps):
            step(us[s % N_DISTINCT], its[s % N_DISTINCT])
        torch.cuda.synchronize()
        torch.use_deterministic_algorithms(prev)
        hashes[K] = {'p': _sha(model.arena), 'loss_sum': step.pop_loss_sum()}
        hashes[K].update({'m': _sha(opt.m), 'v': _sha(opt.v)})
        print(f'hash K={K}: {hashes[K]}', flush=True)
        del model, opt, step
        torch.cuda.empty_cache()
    same = len({json.dumps(h, sort_keys=True) for h in hashes.values()}) == 1

    # ---- timing, arms alternated ----
    arms = {K: _arm(K, dev) for K in lags}
    res = {K: [] for K in lags}

    def ev():
        return torch.cuda.Event(enable_timing=True)

    for r in range(args.rounds):
        for K in (lags if r % 2 == 0 else lags[::-1]):
            model, opt, step = arms[K]
            for s in range(args.warmup):
                step(us[s % N_DISTINCT], its[s % N_DISTINCT])
            a, b = ev(), ev()
            a.record()
            for s in range(args.steps):
                step(us[s % N_DISTINCT], its[s % N_DISTINCT])
            b.record()
            b.synchronize()
            ms_step = a.elapsed_time(b) / args.steps
            tabs, gtabs = model._tables(), opt.grad_tables
            e = [[ev() for _ in range(4)] for _ in range(50)]
            for s in range(50):
                u, i = us[s % N_DISTINCT], its[s % N_DISTINCT]
                e[s][0].record()
                _C.mf_train_fused(tabs, gtabs, u, i, step.kind, step.shift, step.loss_accum, status=model._status())
                e[s][1].record()
                opt.mark(u, i)
                e[s][2].record()
                opt.step_fused()
                e[s][3].record()
            torch.cuda.synchronize()
            k_ms = {name: sum(x[j].elapsed_time(x[j + 1]) for x in e) / 50
                    for j, name in enumerate(('hsk_mf_train_fused', 'hsk_mark_batch', 'adamw'))}
            res[K].append({'ms_step': ms_step, 'kernels_ms': k_ms})
            print(f'round {r} K={K}: step {ms_step:.4f} ms, adamw {k_ms["adamw"]:.4f} ms', flush=True)
            step.pop_loss_sum()
    info['gpu_after'] = gpu_info()

    summary = {}
    for K in lags:
        st = [x['ms_step'] for x in res[K]]
        aw = [x['kernels_ms']['adamw'] for x in res[K]]
        mb = model_bytes(K)
        summary[K] = {'ms_step_median': statistics.median(st), 'ms_step_min': min(st), 'ms_step_max': max(st),
                      'adamw_ms_median': statistics.median(aw), 'adamw_ms_min': min(aw), 'adamw_ms_max': max(aw),
                      'fused_ms_median': statistics.median(x['kernels_ms']['hsk_mf_train_fused'] for x in res[K]),
                      'mark_ms_median': statistics.median(x['kernels_ms']['hsk_mark_batch'] for x in res[K]),
                      'triples_per_s': B * N / (statistics.median(st) * 1e-3),
                      'adamw_model_bytes': mb, 'adamw_model_TBps': mb / (statistics.median(aw) * 1e-3) / 1e12}
    doc = {'what': 'cfg4 training step (FusedMFTrainStep: hsk_mf_train_fused + hsk_mark_batch + one AdamW launch) per '
                   'DenseAdam state_lag; CUDA events, arms alternated in one process',
           'rounds': args.rounds, 'warmup': args.warmup, 'steps': args.steps, 'hash_steps': args.hash_steps,
           'n_params': P + I, 'touched_user_rows_per_step': touched_users, 'touched_item_rows_per_step': touched_items,
           'gpu': info, 'summary': summary, 'runs': res, 'bitwise_equal_p_m_v_loss': same, 'hashes': hashes}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({'summary': summary, 'bitwise_equal_p_m_v_loss': same, 'gpu': info['gpu_before']}, indent=1))


if __name__ == '__main__':
    main()
