"""Cost of the cfg4 optimizer pass, hsk_adamw_dense_rows, for one or more builds of the library.

    python scripts/adamw_cost.py --lib new=hassaku_b200/lib/libhassaku_b200.so --lib old=/path/to/parent/libhassaku_b200.so

Every (label, library) runs in its own process (the library is chosen by HSK_LIB_PATH), and the processes alternate
for --rounds rounds.  Each process:
  * builds the cfg4 arena: 2 M users x 1 M items x d 128 plus the item bias (SGDMatrixFactorization.on_device, seed 64),
    and seeded optimizer state m / v: 40 % of the user rows and 5 % of the item rows never touched (m = v = 0), the
    others with magnitudes of a trained model.  The same in every process;
  * stamps the rows of a real cfg4 batch (bench.make_device_batches on make_device_interactions, hsk_mark_batch) and
    puts a seeded gradient into the stamped rows and the bias vector;
  * on the first round only: runs one pass and hashes p, m, v (identical inputs, no atomics: builds that compute the
    same thing give the same hashes);
  * times hsk_adamw_dense_rows alone: CUDA events around --iters launches after --warmup launches (the 6.2 GB working
    set is far beyond the 126 MB L2, nothing is flushed), and hsk_adamw_dense on the same arena for reference.
Writes --out (JSON) with the card's name, power limit and clocks read in the same run."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

U, I, D, B, N = 2_000_000, 1_000_000, 128, 8192, 50
LR, WD, STEP = 3e-4, 4e-5, 221


def _state(model, dev):
    import torch
    lay = model.layout
    p = model.arena
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    n = p.numel()
    m = torch.randn(n, device=dev, generator=gen) * 1e-5
    m *= torch.exp2(-30 * torch.rand(n, device=dev, generator=gen))        # decayed first moments down to ~1e-14
    v = torch.rand(n, device=dev, generator=gen) * 1e-9 * torch.exp2(-20 * torch.rand(n, device=dev, generator=gen))
    for off, rows, share in ((lay.off_U, lay.n_users, 0.4), (lay.off_V, lay.n_items, 0.05)):
        never = (torch.rand(rows, device=dev, generator=gen) < share).repeat_interleave(lay.ld)
        m[off:off + rows * lay.ld][never] = 0.0
        v[off:off + rows * lay.ld][never] = 0.0
    return p, m, v, gen


def worker(args):
    import torch
    sys.path.insert(0, ROOT)
    from bench import make_device_batches
    from hassaku_b200 import _C
    from hassaku_b200.algorithms.sgd_alg import SGDMatrixFactorization
    from hassaku_b200.data.synthetic import SHAPES, make_device_interactions
    from hassaku_b200.train.optim import stamp_segments
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    _, _, n_inter = SHAPES['lfm2b']
    data = make_device_interactions(U, I, n_inter, dev, 1, 0, seed=0)
    us, its = make_device_batches(data, B, N, 1)
    del data
    model = SGDMatrixFactorization.on_device(U, I, D, use_item_bias=True, device=dev, seed=64)
    lay = model.layout
    p, m, v, gen = _state(model, dev)
    su = torch.zeros(U, dtype=torch.uint8, device=dev)
    si = torch.zeros(I, dtype=torch.uint8, device=dev)
    _C.mark_batch(us[0], its[0], U, I, su, si, STEP)
    segs, su, si = stamp_segments(lay, B, its[0].numel(), su, si)
    g = torch.zeros_like(p)
    for off, rows, ld, st in segs:
        hit = (st[:rows] == _C.row_stamp(STEP)).repeat_interleave(ld)
        g[off:off + rows * ld][hit] = torch.randn(int(hit.sum()), device=dev, generator=gen) * 1e-4
    g[lay.off_Ib:lay.off_Ib + I] = torch.randn(I, device=dev, generator=gen) * 1e-3
    touched_rows = sum(int((st[:rows] == _C.row_stamp(STEP)).sum()) for _, rows, _, st in segs)
    out = {'lib': os.environ.get('HSK_LIB_PATH'), 'n_params': p.numel(), 'touched_rows': touched_rows,
           'rows': U + I, 'segments': len(segs)}

    def rows_pass():
        _C.adamw_dense_rows(p, m, v, g, segs, LR, 0.9, 0.999, 1e-8, WD, STEP, arith=0, adam_l2=False)

    if args.hash:
        rows_pass()
        torch.cuda.synchronize()
        for name, t in (('p', p), ('m', m), ('v', v)):
            h = hashlib.sha256()
            for c in t.view(torch.int32).split(1 << 26):
                h.update(c.cpu().numpy().tobytes())
            out[f'sha256_{name}'] = h.hexdigest()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.iters):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / args.iters

    out['rows_ms'] = timed(rows_pass)
    out['dense_ms'] = timed(lambda: _C.adamw_dense(p, m, v, g, LR, 0.9, 0.999, 1e-8, WD, STEP, arith=0, zero_grad=True))
    print('RESULT ' + json.dumps(out), flush=True)


def gpu_info():
    q = 'name,power.limit,clocks.max.sm,clocks.sm,clocks.mem'
    try:
        r = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], capture_output=True, text=True,
                           timeout=60)
        return dict(zip(q.split(','), [x.strip() for x in r.stdout.splitlines()[0].split(',')]))
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return {'error': str(e)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--lib', action='append', default=[], metavar='LABEL=PATH', help='a build of libhassaku_b200.so')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--iters', type=int, default=100)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'adamw_rows_cost.json'))
    ap.add_argument('--worker', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--hash', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    libs = [x.split('=', 1) for x in args.lib] or [['current', os.path.join(ROOT, 'hassaku_b200', 'lib', 'libhassaku_b200.so')]]
    res = {label: [] for label, _ in libs}
    info = {'gpu_before': gpu_info()}
    for r in range(args.rounds):
        for label, path in (libs if r % 2 == 0 else libs[::-1]):
            cmd = [sys.executable, os.path.abspath(__file__), '--worker', '--warmup', str(args.warmup), '--iters', str(args.iters)]
            if r == 0:
                cmd.append('--hash')
            env = dict(os.environ, HSK_LIB_PATH=os.path.abspath(path))
            p = subprocess.run(cmd, env=env, capture_output=True, text=True)
            line = [x for x in p.stdout.splitlines() if x.startswith('RESULT ')]
            if p.returncode or not line:
                sys.stderr.write(p.stdout + p.stderr)
                raise SystemExit(f'worker {label} failed (exit {p.returncode})')
            d = json.loads(line[0][7:])
            res[label].append(d)
            print(f'round {r} {label}: rows {d["rows_ms"]:.4f} ms, dense {d["dense_ms"]:.4f} ms', flush=True)
    info['gpu_after'] = gpu_info()
    summary = {}
    for label, runs in res.items():
        rows = [x['rows_ms'] for x in runs]
        dense = [x['dense_ms'] for x in runs]
        summary[label] = {'rows_ms_median': statistics.median(rows), 'rows_ms_min': min(rows), 'rows_ms_max': max(rows),
                          'dense_ms_median': statistics.median(dense)}
    base = summary[libs[-1][0]]['rows_ms_median']
    for label in summary:
        summary[label][f'rows_ms_median_over_{libs[-1][0]}'] = summary[label]['rows_ms_median'] / base
    first = res[libs[0][0]][0]
    P = first['n_params']
    hashes = {label: {k: v for k, v in runs[0].items() if k.startswith('sha256')} for label, runs in res.items()}
    same = len({json.dumps(h, sort_keys=True) for h in hashes.values()}) == 1
    doc = {'what': 'hsk_adamw_dense_rows at cfg4 (2 M x 1 M x 128 + item bias, B 8192, N 50, AdamW arith 0), per library '
                   'build; CUDA events around iters launches after warmup launches, processes alternated',
           'rounds': args.rounds, 'warmup': args.warmup, 'iters': args.iters, 'n_params': P,
           'touched_rows': first['touched_rows'], 'rows': first['rows'], 'gpu': info,
           'libs': {label: path for label, path in libs}, 'summary': summary, 'runs': res,
           'bitwise_equal_p_m_v': same, 'hashes': hashes}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({'summary': summary, 'bitwise_equal_p_m_v': same, 'gpu': info['gpu_before']}, indent=1))


if __name__ == '__main__':
    main()
