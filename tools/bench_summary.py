"""Cost of the posterior summaries (quantile / histogram / histogram2d) against a full pass over the cloud.

    python tools/bench_summary.py [--n 100000000] [--reps 20] [--out profiles/summary_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run), each on a broad
cloud (d = 3 normals, explicit random weights) and on a narrow post-resample cloud (the broad cloud weighted by a
narrow Gaussian in every parameter and resampled systematically, so its weights are implicit):
  quantile      quantile(q=(0.025, 0.5, 0.975)) over all parameters
  histogram     histogram(256) over all parameters (range=given, so one pass; the automatic range adds one)
  histogram2d   histogram2d(0, 1, 128)
Each reports the call time (CUDA events around the call, median of --reps; every call ends in one host
synchronisation), the streaming passes it made (obe_summary_passes), and the bytes a pass reads (d rows, plus the
weight row when the weights are explicit) over the per-pass time, next to the device-to-device copy rate measured in
the same run.  host_path: particles + particle_weights + np.quantile(weights=...) of every row, once, at 1e7 and at n.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power = (out[0].split(', ') + ['?'])[:2] if out else ('?', '?')
    return name, power


def copy_rate(torch, nbytes=4 << 30, reps=20):
    a = torch.empty(nbytes // 8, dtype=torch.float64, device='cuda')
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def clouds(obe, torch, n):
    g = torch.Generator(device='cuda').manual_seed(1)
    x = torch.randn((3, n), generator=g, device='cuda', dtype=torch.float64)
    x[1] = x[1] * 300.0 - 1200.0
    x[2] = x[2] * 1e3 + 5e4
    broad = obe.ParticlePDF(np.zeros((3, 1)), seed=1)
    broad.set_pdf(x)
    w = torch.rand(n, generator=g, device='cuda', dtype=torch.float64)
    broad.particle_weights = (w / w.sum()).cpu().numpy()
    narrow = obe.ParticlePDF(np.zeros((3, 1)), seed=2)
    narrow.set_pdf(x)
    z = (x - x.mean(dim=1, keepdim=True)) / x.std(dim=1, keepdim=True)
    lw = -0.5 * ((z - 0.3) / 0.02).pow(2).sum(dim=0)
    w = torch.exp(lw - lw.max())
    narrow.particle_weights = (w / w.sum()).cpu().numpy()
    narrow.resample()
    assert narrow._buf.stats[62].item() > 0, 'the narrow cloud should carry implicit weights'
    return {'broad': broad, 'narrow': narrow}


def time_call(torch, fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=100_000_000)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'summary_b200.jsonl'))
    ap.add_argument('--no-host', action='store_true')
    args = ap.parse_args()
    import torch
    import optbayesexpt_b200 as obe
    assert torch.cuda.is_available(), 'this benchmark needs a CUDA device'
    name, power = card()
    copy = copy_rate(torch)
    n = args.n
    lines = []
    base = dict(card=name, power_limit=power, n=n, d=3, copy_GBps=round(copy, 1))
    for cname, pdf in clouds(obe, torch, n).items():
        explicit = not pdf._buf.stats[62].item() > 0
        lims = [(float(a), float(b)) for a, b in zip(pdf.quantile(0.0)[:, 0], pdf.quantile(1.0)[:, 0])]
        arms = {'quantile': lambda: pdf.quantile((0.025, 0.5, 0.975)),
                'histogram': lambda: pdf.histogram(256, range=lims),
                'histogram2d': lambda: pdf.histogram2d(0, 1, 128, range=lims[:2])}
        for arm, fn in arms.items():
            med, best = time_call(torch, fn, args.reps)
            passes = int(pdf._lib.obe_summary_passes())
            rows = 2 if arm == 'histogram2d' else 3
            per_pass = 8 * n * (rows + (1 if explicit else 0))
            rec = dict(base, arm=arm, cloud=cname, weights='explicit' if explicit else 'implicit',
                       ms=round(med, 4), ms_min=round(best, 4), passes=passes,
                       bytes_per_pass=per_pass, GBps_per_pass=round(per_pass * passes / (med * 1e-3) / 1e9, 1),
                       of_copy=round(per_pass * passes / (med * 1e-3) / 1e9 / copy, 3))
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        del pdf
    if not args.no_host:
        for m in sorted({10_000_000, n}):
            pdf = clouds(obe, torch, m)['broad']
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            x, w = pdf.particles, pdf.particle_weights
            t1 = time.perf_counter()
            np.quantile(x, (0.025, 0.5, 0.975), axis=1, weights=np.broadcast_to(w, x.shape), method='inverted_cdf')
            t2 = time.perf_counter()
            rec = dict(base, n=m, arm='host_path', cloud='broad', copy_s=round(t1 - t0, 3),
                       np_quantile_s=round(t2 - t1, 3), ms=round((t2 - t0) * 1e3, 1))
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            del pdf, x, w
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as f:
        for rec in lines:
            f.write(json.dumps(rec) + '\n')


if __name__ == '__main__':
    main()
