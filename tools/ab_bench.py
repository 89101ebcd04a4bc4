"""A/B timing of two builds of the library on one GPU, alternated so that drift of the card or the host hits both.

    python tools/ab_bench.py A.so B.so OUT_DIR [--rounds 3] [--workloads c1,c3]

Build each side with ``python -m optbayesexpt_b200.build --force --out=<path>``.  Runs
``bench.py --no-cpu-baseline --no-multinomial`` (the c4 flagship) A B A B ... with OBE_B200_LIB selecting the build,
then each extra workload the same way, then ``--dump-outputs`` of c4 for both builds (in a temporary directory) and a
comparison of the dumps.  Writes every bench JSON line to OUT_DIR/ab.jsonl and prints a summary: the card and its power
limit, then per run `value`, `kernels_ms`, `serialised_cycle.kernels_ms` and `sustained`, and the spread per build."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def bench(lib, extra):
    env = dict(os.environ, OBE_B200_LIB=os.path.abspath(lib))
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--no-cpu-baseline', '--no-multinomial'] + extra
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    if res.returncode != 0:
        raise RuntimeError(f'{" ".join(cmd)} failed:\n{res.stdout[-2000:]}\n{res.stderr[-4000:]}')
    lines = [json.loads(x) for x in res.stdout.splitlines() if x.startswith('{')]
    return [x for x in lines if 'value' in x][-1]


def brief(r):
    ser = r.get('serialised_cycle') or {}
    return {'value': r['value'], 'kernels_ms': r.get('kernels_ms'), 'serialised_kernels_ms': ser.get('kernels_ms'),
            'sustained': (r.get('sustained') or {}).get('cycles_per_s')}


def compare_dumps(da, db):
    out = {}
    for f in sorted(os.listdir(da)):
        if not f.endswith('.npy'):
            continue
        a, b = np.load(os.path.join(da, f)), np.load(os.path.join(db, f))
        if a.shape != b.shape:
            out[f] = {'shape': [a.shape, b.shape]}
            continue
        diff = a != b
        den = np.maximum(np.abs(a), np.abs(b))
        rel = np.where(diff, np.abs(a - b) / np.where(den > 0, den, 1.0), 0.0)
        out[f] = {'identical': bool(not diff.any()), 'n_diff': int(diff.sum()), 'size': int(a.size),
                  'max_rel': float(rel.max()) if a.size else 0.0}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('lib_a')
    ap.add_argument('lib_b')
    ap.add_argument('out')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--workloads', default='c1,c3')
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    log = open(os.path.join(args.out, 'ab.jsonl'), 'w')
    sides = {'A': args.lib_a, 'B': args.lib_b}
    print(json.dumps({'card': card(), 'A': args.lib_a, 'B': args.lib_b}), flush=True)
    runs = {'A': [], 'B': []}
    for i in range(args.rounds):
        for s in 'AB':
            r = bench(sides[s], [])
            log.write(json.dumps({'side': s, 'round': i, 'workload': 'c4', 'line': r}) + '\n')
            log.flush()
            runs[s].append(r['value'])
            print(json.dumps({'side': s, 'round': i, 'workload': 'c4', **brief(r)}), flush=True)
    for s in 'AB':
        v = np.array(runs[s])
        print(json.dumps({'side': s, 'c4_mean': v.mean(), 'c4_min': v.min(), 'c4_max': v.max(),
                          'spread': v.max() - v.min()}), flush=True)
    for w in [x for x in args.workloads.split(',') if x]:
        for i in range(args.rounds):
            for s in 'AB':
                r = bench(sides[s], ['--workload', w])
                log.write(json.dumps({'side': s, 'round': i, 'workload': w, 'line': r}) + '\n')
                print(json.dumps({'side': s, 'round': i, 'workload': w, **brief(r)}), flush=True)
    tmp = tempfile.mkdtemp()                      # (the dumps are up to 64 MB each: compared, not kept)
    dumps = {}
    for s in 'AB':
        dumps[s] = os.path.join(tmp, f'dump_{s}')
        bench(sides[s], ['--steps', '3', '--warmup', '2', '--dump-outputs', dumps[s]])
    print(json.dumps({'dump_compare': compare_dumps(dumps['A'], dumps['B'])}), flush=True)
    shutil.rmtree(tmp)
    print(json.dumps({'card_after': card()}), flush=True)


if __name__ == '__main__':
    main()
