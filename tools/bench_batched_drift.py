"""Cost of the batched engines' random-walk drift (BatchedOptBayesExpt(..., drift=...)).

    python tools/bench_batched_drift.py [--instances 4096] [--particles 1e4] [--launches 50] [--cycles 200]
                                        [--rounds 3] [--out profiles/batched_drift_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run):
  pass_d<d>_<shared|per_instance>  obe_batch_drift alone at instances x particles x d (d = 4, 8), one factor for all
                        instances or one per instance, CUDA events around `launches` back-to-back launches (4096 x 1e4
                        x d = 4 is 1.3 GB per buffer, above the 126 MB L2).  Bytes actually moved: the staged weight
                        row and d particle rows over the padded instance (np = whole tiles), plus the d rows written
                        over the live particles: 8 ((1 + d) np + d n) per instance.  The ratio is to the
                        device-to-device copy rate (2 x bytes / time of a 2 GB copy_) measured in the same process.
  loop_c5               closed_loop_cycle of the c5 shape (4096 lock-in instances x 1e4 particles, on-device simulator)
                        with drift=None and with a drift of every parameter, alternated `rounds` times in one process:
                        cycles per second of wall time over `cycles` cycles each, ending in a device synchronise.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power = (out[0].split(', ') + ['?'])[:2] if out else ('?', '?')
    return name, power


def d2d_rate(torch, nbytes=2 << 30, reps=10):
    src = torch.empty(nbytes // 8, dtype=torch.float64, device='cuda').uniform_()
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    del src, dst
    torch.cuda.empty_cache()
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3)


SLOPE = '__device__ void slope(const double* s, const double* p, const double* c, double* y) { y[0] = p[0] * s[0]; }\n'


def _engine(torch, model, B, n, d):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    prior = torch.randn((B, d, n), dtype=torch.float64, device='cuda') + 3.0
    beng = BatchedOptBayesExpt(model, (np.linspace(0.0, 1.0, 5),), prior, (), scale=False, seed=1)
    del prior
    torch.cuda.empty_cache()
    return beng


def pass_arm(torch, model, B, n, d, per_instance, launches, rate):
    from optbayesexpt_b200 import _lib
    from optbayesexpt_b200.drift import batched_drift_factors
    q = np.eye(d) * 1e-4 + 1e-5
    drift = np.broadcast_to(q, (B, d, d)) if per_instance else q
    beng = _engine(torch, model, B, n, d)
    factors = batched_drift_factors(drift, B, d)
    host, dev = beng._factor_args(factors)

    def launch(step):
        _lib.check(beng._lib.obe_batch_drift(beng._bs(), host, beng._ptr(dev), 0, 0, None, 0, 7, step,
                                             beng._stream()))

    for s in range(3):
        launch(s)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(launches):
        launch(100 + s)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    nbytes = 8 * B * ((1 + d) * beng._np + d * n)
    achieved = nbytes / (ms * 1e-3)
    del beng, dev
    torch.cuda.empty_cache()
    return dict(arm=f'pass_d{d}_{"per_instance" if per_instance else "shared"}', instances=B, particles=n, d=d,
                ms=ms, bytes=nbytes, tb_per_s=achieved / 1e12, d2d_tb_per_s=rate / 1e12, ratio_to_d2d=achieved / rate)


def c5_engine(torch, B, n, drift):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    from oracle.scenarios import build_inputs, by_name
    sc = by_name('c5_lockin')
    inp = build_inputs(sc, n)
    g = torch.Generator(device='cuda')
    g.manual_seed(5)
    prior = torch.empty((B, 4, n), dtype=torch.float64, device='cuda')
    scales = (1e-3, 10.0, 1e-5, 10.0)
    for j, s in enumerate(scales):
        prior[:, j] = torch.empty((B, n), dtype=torch.float64, device='cuda').exponential_(1.0, generator=g) * s
    beng = BatchedOptBayesExpt('lockin_coil', inp['setting_values'], prior, (), noise_parameter_index=(3, 3),
                               constraint_lt=(0, 1, 2, 3), cost_of_changing_setting=5.0, scale=False, seed=11,
                               drift=[1e-3 * s for s in scales] if drift else None)
    del prior
    beng.set_simulator(np.tile(sc['true_pars'], (B, 1)), 5.0, seed=3)
    return beng


def loop_c5(torch, B, n, cycles, rounds):
    engines = {drift: c5_engine(torch, B, n, drift) for drift in (False, True)}
    per_s = {False: [], True: []}
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for beng in engines.values():
            for _ in range(20):
                beng.closed_loop_cycle()
        torch.cuda.synchronize()
        for _ in range(rounds):
            for drift, beng in engines.items():
                t0 = time.perf_counter()
                for _ in range(cycles):
                    beng.closed_loop_cycle()
                torch.cuda.synchronize()
                per_s[drift].append(cycles / (time.perf_counter() - t0))
    return dict(arm='loop_c5', instances=B, particles=n, cycles=cycles, rounds=rounds,
                per_s_without=per_s[False], per_s_with_drift=per_s[True],
                median_without=float(np.median(per_s[False])), median_with_drift=float(np.median(per_s[True])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--instances', type=int, default=4096)
    ap.add_argument('--particles', type=float, default=1e4)
    ap.add_argument('--launches', type=int, default=50)
    ap.add_argument('--cycles', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'batched_drift_b200.jsonl'))
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'this benchmark needs a CUDA device'
    from optbayesexpt_b200.models import cuda_source
    name, power = card()
    model = cuda_source(SLOPE, 'slope', 1, 1)        # one parameter in the model, any number of rows in the cloud
    B, n = args.instances, int(args.particles)
    rows = []
    for d in (4, 8):
        for per_instance in (False, True):
            rate = d2d_rate(torch)
            rows.append(pass_arm(torch, model, B, n, d, per_instance, args.launches, rate))
            print(json.dumps(rows[-1]), flush=True)
    rows.append(loop_c5(torch, B, n, args.cycles, args.rounds))
    print(json.dumps(rows[-1]), flush=True)
    out = args.out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, 'w') as f:
        for r in rows:
            r.update(gpu=name, power_limit=power)
            f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
