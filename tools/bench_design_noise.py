"""Cost and effect of the likelihood-aware utility (design_noise='likelihood').

    python tools/bench_design_noise.py [--launches 200] [--rounds 5] [--cycles 300] [--seeds 16] [--steps 150]
                                       [--out profiles/design_noise_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run):
  utility_<lik>_<S>     the utility kernel (obe_utility, variance method, K = 30) of a non-Gaussian handle over S
                        settings, 'fixed' against 'likelihood': CUDA events around `launches` back-to-back launches of
                        the C entry, the two modes alternated `rounds` times; the median per-launch time of each mode.
                        Poisson: lorentzian_hwhm as rates; binomial: lorentzian_dip as probabilities.
  c3_poisson_<mode>     rabi, 1e6 particles x 101^2 settings, Poisson counts, pdf_update + opt_setting with the
                        resample test on the device, natural resample rate: cycles/s (modes alternated, two runs each).
  study_peak            a Poisson Lorentzian peak on a background (lorentzian_hwhm, 1e5 particles, 241 settings),
                        `seeds` simulated experiments of `steps` measurements per mode: the median final posterior std
                        of the peak position.  'fixed' uses default_noise_std = 5 counts (about sqrt of the mean count).
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


def utility_engines(obe, lik, n_settings):
    """A 'fixed' and a 'likelihood' engine on one model with the same draws already on the device."""
    g = np.random.default_rng(1)
    n = 100_000
    if lik == 'poisson':
        model, cons, aux = obe.builtin('lorentzian_hwhm'), (0.3,), None
        prior = np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(2.0, 10.0, n)])
    else:
        model, cons, aux = obe.builtin('lorentzian_dip'), (), 100.0
        prior = np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 0.8, n), g.uniform(0.2, 0.6, n)])
    s = (np.linspace(1.5, 4.5, n_settings),)
    engines = {}
    for mode in ('fixed', 'likelihood'):
        e = obe.OptBayesExpt(model, s, prior, cons, likelihood_model=lik, design_noise=mode, design_aux=aux,
                             default_noise_std=5.0 if lik == 'poisson' else 0.05)
        e.rng = np.random.default_rng(2)
        e._randdraw_dev(30, out=e._draws_buffer())
        engines[mode] = e
    return engines


def utility_args(e):
    from optbayesexpt_b200 import _lib
    n_set = len(e.setting_indices)
    vn = _lib.darr(np.asarray(e._design_var_noise(), dtype=np.float64).reshape(-1), _lib.MAX_CHANNELS)
    return (e._model, C.c_void_p(e._draws_buffer().data_ptr()), 30, C.c_void_p(e._settings_dev.data_ptr()), e._lds,
            n_set, e._cons_arr, vn, None, None, 0, 0, None, C.c_void_p(e._utility_dev.data_ptr()),
            C.c_void_p(e._best_dev.data_ptr()), C.c_void_p(e._select_scratch.data_ptr()), e._stream())


def time_launches(torch, lib, args, launches):
    from optbayesexpt_b200 import _lib
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        _lib.check(lib.obe_utility(*args))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def utility_arm(obe, torch, lik, n_settings, launches, rounds):
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    engines = utility_engines(obe, lik, n_settings)
    args = {m: utility_args(e) for m, e in engines.items()}
    for m in args:                                      # warm-up (module load, shared-memory opt-in)
        time_launches(torch, lib, args[m], 20)
    ms = {m: [] for m in args}
    for _ in range(rounds):
        for m in ('fixed', 'likelihood'):
            ms[m].append(time_launches(torch, lib, args[m], launches))
    med = {m: float(np.median(v)) for m, v in ms.items()}
    return med, ms


def c3_arm(obe, mode, cycles, warmup=20):
    import torch

    from oracle import obe_oracle as orc
    from oracle.scenarios import build_inputs, by_name
    sc = by_name('c3_pipulse')
    inp = build_inputs(sc, 1_000_000)
    eng = obe.OptBayesExpt('rabi', inp['setting_values'], inp['prior'], inp['cons'], scale=False,
                           default_noise_std=300.0, likelihood_model='poisson', design_noise=mode, seed=3)
    eng.eager_select = eng.async_update = True
    meas = np.random.default_rng(1002)
    fired = 0

    def step(x):
        mu = orc.model_rabi(x, sc['true_pars'], inp['cons'])
        eng.pdf_update((x, float(meas.poisson(mu))))
        return eng.opt_setting()

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


def study_arm(obe, mode, seeds, steps):
    """Median final posterior std of the peak position over `seeds` simulated Poisson experiments."""
    from oracle import obe_oracle as orc
    truth, cons, n = (3.1, 40.0, 10.0), (0.3,), 100_000
    s = (np.linspace(0.0, 6.0, 241),)
    model = obe.builtin('lorentzian_hwhm')
    stds = []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for seed in range(seeds):
            g = np.random.default_rng(100 + seed)
            prior = np.array([g.uniform(1.0, 5.0, n), g.uniform(10.0, 80.0, n), g.uniform(2.0, 20.0, n)])
            eng = obe.OptBayesExpt(model, s, prior, cons, likelihood_model='poisson', design_noise=mode,
                                   default_noise_std=5.0, seed=200 + seed)
            eng.rng = np.random.default_rng(300 + seed)
            meas = np.random.default_rng(400 + seed)
            for _ in range(steps):
                x = eng.opt_setting()
                eng.pdf_update((x, float(meas.poisson(orc.model_lorentzian_hwhm(x, truth, cons)))))
            stds.append(float(eng.std()[0]))
    return float(np.median(stds)), stds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--cycles', type=int, default=300)
    ap.add_argument('--seeds', type=int, default=16)
    ap.add_argument('--steps', type=int, default=150)
    ap.add_argument('--sizes', default='10000,100000,1000000')
    ap.add_argument('--out', default=os.path.join('profiles', 'design_noise_b200.jsonl'))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_design_noise.py measures on a CUDA device; none is visible')
    import optbayesexpt_b200 as obe
    name, power = card()
    base = dict(gpu=name, power_limit=power)
    lines = []

    def emit(d):
        lines.append(dict(base, **d))
        print(json.dumps(lines[-1]), flush=True)

    for lik in ('poisson', 'binomial'):
        for n_settings in (int(v) for v in a.sizes.split(',')):
            med, ms = utility_arm(obe, torch, lik, n_settings, a.launches, a.rounds)
            emit(dict(arm=f'utility_{lik}_{n_settings}', likelihood=lik, n_settings=n_settings, n_draws=30,
                      launches=a.launches, rounds=a.rounds, fixed_us=round(1e3 * med['fixed'], 2),
                      likelihood_us=round(1e3 * med['likelihood'], 2),
                      ratio=round(med['likelihood'] / med['fixed'], 3),
                      fixed_us_rounds=[round(1e3 * v, 2) for v in ms['fixed']],
                      likelihood_us_rounds=[round(1e3 * v, 2) for v in ms['likelihood']]))
    rates = {'fixed': [], 'likelihood': []}
    fired = {'fixed': [], 'likelihood': []}
    for _ in range(2):
        for mode in ('fixed', 'likelihood'):
            r, f = c3_arm(obe, mode, a.cycles)
            rates[mode].append(round(r, 1))
            fired[mode].append(f)
    for mode in ('fixed', 'likelihood'):
        emit(dict(arm=f'c3_poisson_{mode}', model='rabi', likelihood='poisson', design_noise=mode, n=1_000_000,
                  n_settings=101 * 101, cycles=a.cycles, resamples=fired[mode], cycles_per_s_runs=rates[mode],
                  cycles_per_s=float(np.median(rates[mode]))))
    lines[-1]['vs_fixed'] = round(lines[-1]['cycles_per_s'] / lines[-2]['cycles_per_s'], 3)
    study = {}
    for mode in ('fixed', 'likelihood'):
        study[mode] = study_arm(obe, mode, a.seeds, a.steps)
    emit(dict(arm='study_peak', model='lorentzian_hwhm', likelihood='poisson', truth=[3.1, 40.0, 10.0],
              n=100_000, n_settings=241, seeds=a.seeds, steps=a.steps, default_noise_std=5.0,
              median_std_x0_fixed=round(study['fixed'][0], 5), median_std_x0_likelihood=round(study['likelihood'][0], 5),
              std_x0_fixed=[round(v, 5) for v in study['fixed'][1]],
              std_x0_likelihood=[round(v, 5) for v in study['likelihood'][1]]))
    os.makedirs(os.path.dirname(a.out) or '.', exist_ok=True)
    with open(a.out, 'w') as f:
        for ln in lines:
            f.write(json.dumps(ln) + '\n')
    print('wrote', a.out)


if __name__ == '__main__':
    main()
