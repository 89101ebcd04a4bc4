"""Cost and effect of the information gain of a user count likelihood (cuda_likelihood(..., window=)).

    python tools/bench_information_gain_user.py [--launches 100] [--rounds 3] [--seeds 16] [--steps 150]
                                                [--out profiles/information_gain_user_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run):
  poisson_<level>       method 4 over 1e4 settings, K = 30, broad draws of lorentzian_hwhm as rates at a mean count
                        `level` (1, 100): the built-in Poisson design handle against the same Poisson restated as a
                        user pmf with the built-in's windows (oracle/count_pmfs.py), on the same draws, CUDA events
                        around back-to-back launches of the C entry, the two alternated `rounds` times; the median
                        per-launch time, and ns per term with terms = K |union of windows| summed over the settings.
  <pmf>                 the same for the negative binomial (r = 20, rates of 2 .. 90), the two-Poisson readout
                        (lam_d = 0.5, lam_b = 3) and the beta-binomial (n = 40) over lorentzian_dip probabilities.
  study                 lorentzian_dip as P(bright) with single-shot readout (lam_d = 0.5, lam_b = 3), 1e5 particles,
                        `seeds` experiments of `steps` measurements per mode: the median final posterior std of every
                        parameter under 'information_gain' and under the 'likelihood' variance utility (noise_var of
                        the mixture).
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

K, S = 30, 10_000


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power = (out[0].split(', ') + ['?'])[:2] if out else ('?', '?')
    return name, power


def engine(obe, lik, model, prior, cons, aux):
    e = obe.OptBayesExpt(obe.builtin(model), (np.linspace(1.5, 4.5, S),), prior, cons, likelihood_model=lik,
                         design_noise='likelihood', design_aux=aux, utility_method='information_gain')
    e.rng = np.random.default_rng(2)
    e._randdraw_dev(K, out=e._draws_buffer())
    return e


def utility_args(e, draws):
    from optbayesexpt_b200 import _lib
    vn = _lib.darr(np.asarray(e._design_var_noise(), dtype=np.float64).reshape(-1), _lib.MAX_CHANNELS)
    return (e._model, C.c_void_p(draws.data_ptr()), K, C.c_void_p(e._settings_dev.data_ptr()), e._lds, S,
            e._cons_arr, vn, None, None, 4, 0, None, C.c_void_p(e._utility_dev.data_ptr()),
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


def terms(e, draws, window, aux):
    from oracle import information_gain as oig
    d = draws.cpu().numpy()
    ys = np.stack([e.eval_over_all_settings(d[:, j]) for j in range(K)]).reshape(K, -1)
    return float(sum(K * len(oig.union_counts(*window(ys[:, s], aux))) for s in range(S)))


def kernel_arm(obe, torch, arms, launches, rounds):
    """arms: {name: (engine, window twin, aux)} sharing one draws buffer; alternated, median ms per launch"""
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    first = next(iter(arms.values()))[0]
    draws = first._draws_buffer()
    args = {n: utility_args(e, draws) for n, (e, _, _) in arms.items()}
    for a in args.values():
        time_launches(torch, lib, a, 3)
    ms = {n: [] for n in args}
    for _ in range(rounds):
        for n, a in args.items():
            ms[n].append(time_launches(torch, lib, a, launches))
    out = {}
    for n, (e, win, aux) in arms.items():
        t = terms(e, draws, win, aux)
        med = float(np.median(ms[n]))
        out[n] = dict(ms=med, ms_rounds=ms[n], terms=t, ns_per_term=med * 1e6 / t)
    return out


def study(obe, seeds, steps):
    from oracle import count_pmfs as cp
    from oracle.obe_oracle import model_lorentzian_dip
    src, entry, nv, win = cp.pmf('readout', lam_d=0.5, lam_b=3.0)[:4]
    lik = obe.cuda_likelihood(src, entry, noise_var=nv, window=win)
    truth = (3.1, 0.6, 0.35)
    settings = (np.linspace(1.5, 4.5, 241),)
    res = {}
    for mode in ('information_gain', 'variance_approx'):
        finals, t0 = [], time.time()
        for seed in range(seeds):
            g = np.random.default_rng(100 + seed)
            n = 100_000
            prior = np.array([g.uniform(2.0, 4.0, n), g.uniform(0.0, 1.0, n), g.uniform(0.2, 0.6, n)])
            e = obe.OptBayesExpt(obe.builtin('lorentzian_dip'), settings, prior, (), likelihood_model=lik,
                                 design_noise='likelihood', utility_method=mode, seed=seed)
            e.rng = np.random.default_rng(seed)
            meas = np.random.default_rng(10_000 + seed)
            for _ in range(steps):
                x = e.opt_setting()
                p = float(model_lorentzian_dip((x[0],), truth, ()))
                c = float(meas.poisson(3.0 if meas.random() < p else 0.5))
                e.pdf_update((x, c, 1.0))
            finals.append(np.asarray(e.std()).reshape(-1))
        res[mode] = dict(median_std=np.median(finals, axis=0).tolist(), seconds=time.time() - t0)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=100)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--seeds', type=int, default=16)
    ap.add_argument('--steps', type=int, default=150)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'information_gain_user_b200.jsonl'))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_information_gain_user needs a CUDA device')
    import optbayesexpt_b200 as obe
    from oracle import count_pmfs as cp
    name, power = card()
    lines = []
    warnings.simplefilter('ignore', RuntimeWarning)
    g = np.random.default_rng(1)
    n = 100_000
    for level in (1.0, 100.0):
        prior = np.array([g.uniform(2.0, 4.0, n), g.uniform(0.4 * level, 1.6 * level, n),
                          g.uniform(0.05 * level, 0.3 * level, n)])
        src, entry, nv, win, _, _, win_np = cp.pmf('poisson')
        arms = {'builtin': (engine(obe, 'poisson', 'lorentzian_hwhm', prior, (0.3,), None), cp.poisson_window, 1.0),
                'user': (engine(obe, obe.cuda_likelihood(src, entry, noise_var=nv, window=win), 'lorentzian_hwhm',
                                prior, (0.3,), None), win_np, 1.0)}
        r = kernel_arm(obe, torch, arms, a.launches, a.rounds)
        lines.append(dict(arm=f'poisson_{level:g}', settings=S, k=K, **{f'{m}_{k}': v for m, d in r.items()
                                                                       for k, v in d.items()},
                          user_over_builtin=r['user']['ms'] / r['builtin']['ms']))
        print(json.dumps(lines[-1]), flush=True)
    peak = np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(2.0, 10.0, n)])
    dip = np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 0.8, n), g.uniform(0.2, 0.6, n)])
    for pmf, model, prior, cons, aux in (('negbin', 'lorentzian_hwhm', peak, (0.3,), 20.0),
                                         ('readout', 'lorentzian_dip', dip, (), 1.0),
                                         ('betabinom', 'lorentzian_dip', dip, (), 40.0)):
        src, entry, nv, win, _, _, win_np = cp.pmf(pmf)
        e = engine(obe, obe.cuda_likelihood(src, entry, noise_var=nv, window=win), model, prior, cons, aux)
        r = kernel_arm(obe, torch, {pmf: (e, win_np, aux)}, a.launches, a.rounds)[pmf]
        lines.append(dict(arm=pmf, settings=S, k=K, **r))
        print(json.dumps(lines[-1]), flush=True)
    if a.seeds > 0:
        lines.append(dict(arm='study', seeds=a.seeds, steps=a.steps, particles=100_000,
                          params=['f0', 'A', 'lw'], **study(obe, a.seeds, a.steps)))
        print(json.dumps(lines[-1]), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        for ln in lines:
            f.write(json.dumps(dict(card=name, power_limit=power, **ln)) + '\n')


if __name__ == '__main__':
    main()
