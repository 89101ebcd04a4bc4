"""Cost of the non-Gaussian likelihoods on the update kernel and on a closed loop.

    python tools/bench_likelihood.py [--n 100000000] [--launches 60] [--cycles 300] [--out profiles/likelihood.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run):
  update_gaussian / update_poisson   lorentzian_hwhm, d = 3, n particles: the model-evaluating update kernel,
  update_binomial                    lorentzian_dip as a probability.  All three stream 8 (d + 2) bytes per
                                     particle (weights in and out, d rows in); GB/s is that over the mean kernel time,
                                     next to the device-to-device copy rate measured in the same run.
  c3_gaussian / c3_poisson           rabi, 1e6 particles x 101^2 settings, pdf_update + opt_setting with the resample
                                     test on the device, natural resample rate: cycles/s.
The update timings are CUDA events around back-to-back launches of the C entry (no host synchronisation between).
The 1e8-particle cloud (2.4 GB of particles) is far larger than the L2, so every launch streams from HBM.
"""
import argparse
import ctypes as C
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


def update_arm(obe, torch, model, likelihood, n, launches, rec):
    from optbayesexpt_b200 import _lib
    g = torch.Generator(device='cuda').manual_seed(1)
    if model == 'lorentzian_hwhm':
        lo, hi = torch.tensor([2.0, -2000.0, 49000.0]), torch.tensor([4.0, -400.0, 51000.0])
        cons = (0.1,)
    else:
        lo, hi = torch.tensor([2.0, 0.2, 0.2]), torch.tensor([4.0, 0.8, 0.6])
        cons = ()
    prior = lo[:, None].cuda() + (hi - lo)[:, None].cuda() * torch.rand((3, n), generator=g, device='cuda',
                                                                         dtype=torch.float64)
    eng = obe.OptBayesExpt(model, (np.linspace(1.5, 4.5, 64),), prior, cons, likelihood_model=likelihood,
                           default_noise_std=500.0)
    del prior
    lib = _lib.load()
    y, sig, _, n_lik = eng._likelihood_spec(rec)
    args = (eng._model, eng._cs(), _lib.darr(rec[0], _lib.MAX_SETTINGS), eng._cons_arr, _lib.darr(y, _lib.MAX_CHANNELS),
            None if sig is None else _lib.darr(sig, _lib.MAX_CHANNELS), None, n_lik, 0, 0.0,
            _lib.darr(eng._pivot, _lib.MAX_PARAMS), eng._stream())
    for _ in range(5):
        _lib.check(lib.obe_update(*args))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        _lib.check(lib.obe_update(*args))
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    del eng
    torch.cuda.empty_cache()
    return ms


def c3_arm(obe, likelihood, cycles, warmup=20):
    from oracle import obe_oracle as orc
    from oracle.scenarios import build_inputs, by_name
    sc = by_name('c3_pipulse')
    inp = build_inputs(sc, 1_000_000)
    eng = obe.OptBayesExpt('rabi', inp['setting_values'], inp['prior'], inp['cons'], scale=False,
                           default_noise_std=300.0, likelihood_model=likelihood, seed=3)
    eng.eager_select = eng.async_update = True
    meas = np.random.default_rng(1002)
    fired = 0

    def step(x):
        mu = orc.model_rabi(x, sc['true_pars'], inp['cons'])
        if likelihood == 'poisson':
            eng.pdf_update((x, float(meas.poisson(mu))))
        else:
            y = mu + np.sqrt(mu) * meas.standard_normal()
            eng.pdf_update((x, float(y), float(np.sqrt(abs(y)))))
        return eng.opt_setting()

    import torch
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        x = eng.opt_setting()
        for _ in range(warmup):
            x = step(x)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(cycles):
            x = step(x)
            fired += int(eng.just_resampled)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    return cycles / dt, fired


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=100_000_000)
    ap.add_argument('--launches', type=int, default=60)
    ap.add_argument('--cycles', type=int, default=300)
    ap.add_argument('--out', default=os.path.join('profiles', 'likelihood_b200.jsonl'))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_likelihood.py measures on a CUDA device; none is visible')
    import optbayesexpt_b200 as obe
    name, power = card()
    peak = copy_rate(torch)
    lines = []
    base = dict(gpu=name, power_limit=power, d2d_copy_gbs=round(peak, 1))
    d = 3
    bpp = 8 * (d + 2)
    arms = [('update_gaussian', 'lorentzian_hwhm', 'gaussian', ((3.0,), 49800.0, 500.0)),
            ('update_poisson', 'lorentzian_hwhm', 'poisson', ((3.0,), 49800.0)),
            ('update_binomial', 'lorentzian_dip', 'binomial', ((3.0,), 61.0, 100.0))]
    for arm, model, lik, rec in arms:
        ms = update_arm(obe, torch, model, lik, a.n, a.launches, rec)
        gbs = bpp * a.n / (ms * 1e-3) / 1e9
        lines.append(dict(base, arm=arm, model=model, likelihood=lik, n=a.n, d=d, launches=a.launches,
                          bytes_per_particle=bpp, kernel_ms=round(ms, 4), gbs=round(gbs, 1),
                          share_of_copy_rate=round(gbs / peak, 3)))
        print(json.dumps(lines[-1]), flush=True)
    g_ms = lines[0]['kernel_ms']
    for ln in lines[1:]:
        ln['vs_gaussian'] = round(ln['kernel_ms'] / g_ms, 3)
    for arm, lik in (('c3_gaussian', 'gaussian'), ('c3_poisson', 'poisson')):
        rate, fired = c3_arm(obe, lik, a.cycles)
        lines.append(dict(base, arm=arm, model='rabi', likelihood=lik, n=1_000_000, n_settings=101 * 101,
                          cycles=a.cycles, resamples=fired, cycles_per_s=round(rate, 1)))
        print(json.dumps(lines[-1]), flush=True)
    lines[-1]['vs_gaussian'] = round(lines[-1]['cycles_per_s'] / lines[-2]['cycles_per_s'], 3)
    os.makedirs(os.path.dirname(a.out) or '.', exist_ok=True)
    with open(a.out, 'w') as f:
        for ln in lines:
            f.write(json.dumps(ln) + '\n')
    print('wrote', a.out)


if __name__ == '__main__':
    main()
