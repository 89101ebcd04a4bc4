"""Cost of the random-walk drift (OptBayesExpt(..., drift=...)).

    python tools/bench_drift.py [--particles 1e8] [--launches 20] [--steps 20] [--cycles 300]
                                [--out profiles/drift_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run):
  pass_d<d>_<weights>   obe_drift alone at `particles` x d (3, 8), explicit or implicit weights, CUDA events around
                        `launches` back-to-back launches; bytes = (16 d + 8) N explicit, 16 d N implicit (every row
                        drifts: read and written once, the weight row read once); the ratio to the device-to-device
                        copy rate (2 x bytes / time of a 2 GB copy_) measured right before, in the same process.
  cycle_<kind>          run_cycle_async at `particles` (Lorentzian, 1e4 settings, K = 30), kind = plain (no resample)
                        or forced (resample every cycle), with and without drift: ms per cycle over `steps` cycles.
  loop_<c1|c3>          the c1 / c3 demo shapes (1e4 particles), closed loop opt_setting + pdf_update with the resample
                        test on the device (eager_select, async_update), with and without drift: cycles per second
                        of wall time over `cycles` cycles after 30 warm-up cycles.
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
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3)


def pass_arm(obe, torch, n, d, implicit, launches):
    import ctypes as C
    from optbayesexpt_b200 import _lib
    prior = torch.randn((d, n), dtype=torch.float64, device='cuda') + 3.0
    pdf = obe.ParticlePDF(prior, seed=1)
    del prior
    if implicit:
        pdf.resample()
        pdf._alt = None
    else:
        pdf._buf.weights[:n].uniform_()
        pdf._buf.stats[_lib.ST_UNIFORM] = 0.0
        pdf._refresh()
    torch.cuda.empty_cache()
    factor = _lib.darr(np.linalg.cholesky(np.eye(d) * 1e-4 + 1e-5).reshape(-1))
    pivot = _lib.darr(np.full(d, 3.0), _lib.MAX_PARAMS)

    def launch(epoch):
        _lib.check(pdf._lib.obe_drift(pdf._cs(), factor, 0, 0, None, 0, pivot, 7, epoch, None, pdf._stream()))

    for ep in range(3):
        launch(ep)
    rate = d2d_rate(torch)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for ep in range(launches):
        launch(100 + ep)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    nbytes = (16 * d if implicit else 16 * d + 8) * n
    achieved = nbytes / (ms * 1e-3)
    del pdf
    torch.cuda.empty_cache()
    return dict(arm=f'pass_d{d}_{"implicit" if implicit else "explicit"}', particles=n, d=d, ms=ms, bytes=nbytes,
                tb_per_s=achieved / 1e12, d2d_tb_per_s=rate / 1e12, ratio_to_d2d=achieved / rate)


def cycle_arm(obe, torch, n, steps, forced, drift):
    prior = torch.stack([torch.rand(n, dtype=torch.float64, device='cuda') * 2 + 2,
                         torch.rand(n, dtype=torch.float64, device='cuda') * -1600 - 400,
                         torch.randn(n, dtype=torch.float64, device='cuda') * 1000 + 50000])
    eng = obe.OptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 10_000),), prior, (0.1,), scale=False,
                           default_noise_std=500.0, seed=3, drift=[1e-3, 0.0, 0.0] if drift else None)
    del prior
    rec = ((3.0,), 49500.0, 5e4)
    for _ in range(3):
        eng.run_cycle_async(rec, resample=forced, select=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        eng.run_cycle_async(rec, resample=forced, select=True)
    e1.record()
    torch.cuda.synchronize()
    del eng
    torch.cuda.empty_cache()
    return e0.elapsed_time(e1) / steps


def loop_arm(obe, name, cycles, drift):
    from oracle import obe_oracle as orc
    from oracle.scenarios import build_inputs, by_name
    sc = by_name(name)
    inp = build_inputs(sc)
    model = getattr(orc, 'model_' + sc['model'])
    eng = obe.OptBayesExpt(sc['model'], inp['setting_values'], inp['prior'], inp['cons'], scale=False,
                           default_noise_std=sc['default_noise_std'], seed=3,
                           drift=(0.002 * inp['prior'].std(axis=1)) if drift else None)
    eng.eager_select = eng.async_update = True
    meas = np.random.default_rng(4)

    def one():
        x = eng.opt_setting()
        mu = float(np.asarray(model(x, sc['true_pars'], inp['cons'])).reshape(-1)[0])
        sig = float(np.sqrt(abs(mu))) if sc['noise'] == 'sqrt' else float(sc['noise'])
        eng.pdf_update((x, mu + sig * float(meas.normal()), sig))

    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(30):
            one()
        fired = 0
        t0 = time.perf_counter()
        for _ in range(cycles):
            one()
            fired += int(eng.just_resampled)
        eng.opt_setting()
        dt = time.perf_counter() - t0
    return cycles / dt, fired


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--particles', type=float, default=1e8)
    ap.add_argument('--launches', type=int, default=20)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--cycles', type=int, default=300)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'drift_b200.jsonl'))
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'this benchmark needs a CUDA device'
    import optbayesexpt_b200 as obe
    name, power = card()
    n = int(args.particles)
    rows = []
    for d in (3, 8):
        for implicit in (False, True):
            rows.append(pass_arm(obe, torch, n, d, implicit, args.launches))
            print(json.dumps(rows[-1]), flush=True)
    for forced in (False, True):
        ms = {drift: cycle_arm(obe, torch, n, args.steps, forced, drift) for drift in (False, True)}
        rows.append(dict(arm=f'cycle_{"forced" if forced else "plain"}', particles=n, ms_without=ms[False],
                         ms_with_drift=ms[True]))
        print(json.dumps(rows[-1]), flush=True)
    for sc in ('c1_find_peak', 'c3_pipulse'):
        res = {drift: loop_arm(obe, sc, args.cycles, drift) for drift in (False, True)}
        rows.append(dict(arm=f'loop_{sc[:2]}', cycles=args.cycles, per_s_without=res[False][0],
                         per_s_with_drift=res[True][0], resamples_without=res[False][1],
                         resamples_with_drift=res[True][1]))
        print(json.dumps(rows[-1]), flush=True)
    out = args.out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, 'w') as f:
        for r in rows:
            r.update(gpu=name, power_limit=power)
            f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
