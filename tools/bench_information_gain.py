"""Cost and effect of the information-gain utility (utility_method='information_gain').

    python tools/bench_information_gain.py [--launches 200] [--rounds 3] [--cycles 300] [--info-cycles 30]
                                           [--seeds 16] [--steps 150] [--out profiles/information_gain_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run):
  utility_<lik>_<level>_<prior>_<S>  the utility kernel of one likelihood-aware design handle (K = 30) over S
                        settings: method 4 (information gain) against method 0 (the 'likelihood' variance utility) on
                        the same draws, CUDA events around `launches` back-to-back launches of the C entry, the two
                        methods alternated `rounds` times; the median per-launch time of each.  Poisson: lorentzian_hwhm
                        as rates at a mean count `level` (1, 100, 1e4); binomial: lorentzian_dip as probabilities with
                        n = `level` trials (10, 1000).  `terms_per_setting`: the mean of K |union of windows| over the
                        grid (the pmf terms the kernel sums), from the draws' outputs.
  c3_<mode>             rabi, 1e6 particles x 101^2 settings, Poisson counts (the c3 scenario, up to 1e5 counts),
                        pdf_update + opt_setting with the resample test on the device, natural resample rate:
                        cycles/s, the 'likelihood' variance utility against the information gain, alternated, two runs
                        each (`info_cycles` cycles for the information gain: its cost grows with the counts).
  study_<counts>        a Poisson Lorentzian peak on a background (lorentzian_hwhm, 1e5 particles, 241 settings),
                        `seeds` simulated experiments of `steps` measurements per mode at the original counts
                        (a = 40, b = 10) and at low counts (a = 4, b = 1): the median final posterior std of every
                        parameter for 'fixed' (default_noise_std = 5), 'likelihood' (variance) and 'information_gain'.
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


def utility_engine(obe, lik, level, prior_kind, n_settings):
    """An information-gain engine with K = 30 draws already on the device."""
    g = np.random.default_rng(1)
    n = 100_000
    tight = prior_kind == 'tight'

    def u(lo, hi, c):
        return c * (1.0 + 1e-3 * g.standard_normal(n)) if tight else g.uniform(lo, hi, n)
    if lik == 'poisson':                                 # peak a on background b: counts between b and a + b
        model, cons, aux = obe.builtin('lorentzian_hwhm'), (0.3,), None
        prior = np.array([u(2.0, 4.0, 3.0), u(0.4 * level, 1.6 * level, level), u(0.05 * level, 0.3 * level,
                                                                                 0.2 * level)])
    else:
        model, cons, aux = obe.builtin('lorentzian_dip'), (), float(level)
        prior = np.array([u(2.0, 4.0, 3.0), u(0.2, 0.8, 0.5), u(0.2, 0.6, 0.4)])
    s = (np.linspace(1.5, 4.5, n_settings),)
    e = obe.OptBayesExpt(model, s, prior, cons, likelihood_model=lik, design_noise='likelihood', design_aux=aux,
                         utility_method='information_gain')
    e.rng = np.random.default_rng(2)
    e._randdraw_dev(30, out=e._draws_buffer())
    return e


def terms_per_setting(e, lik, level, sample=400):
    from oracle import information_gain as oig
    draws = e._draws_buffer().cpu().numpy()
    ys = np.stack([e.eval_over_all_settings(draws[:, j])[0] for j in range(draws.shape[1])])
    idx = np.linspace(0, ys.shape[1] - 1, min(sample, ys.shape[1])).astype(int)
    n = float(level) if lik == 'binomial' else None
    counts = [ys.shape[0] * len(oig.union_counts(*oig.windows(ys[:, i], lik, n))) for i in idx]
    return float(np.mean(counts))


def utility_args(e, method):
    from optbayesexpt_b200 import _lib
    n_set = len(e.setting_indices)
    vn = _lib.darr(np.asarray(e._design_var_noise(), dtype=np.float64).reshape(-1), _lib.MAX_CHANNELS)
    return (e._model, C.c_void_p(e._draws_buffer().data_ptr()), 30, C.c_void_p(e._settings_dev.data_ptr()), e._lds,
            n_set, e._cons_arr, vn, None, None, method, 0, None, C.c_void_p(e._utility_dev.data_ptr()),
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


def utility_arm(obe, torch, lik, level, prior_kind, n_settings, launches, rounds):
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    e = utility_engine(obe, lik, level, prior_kind, n_settings)
    args = {'variance': utility_args(e, 0), 'information_gain': utility_args(e, 4)}
    # `launches` launches, or as many as fill about a second for the slow (high-count) arms
    probe = time_launches(torch, lib, args['information_gain'], 3)
    n_launch = int(max(5, min(launches, 1000.0 / max(probe, 1e-3))))
    for m in args:
        time_launches(torch, lib, args[m], 5)
    ms = {m: [] for m in args}
    for _ in range(rounds):
        for m in args:
            ms[m].append(time_launches(torch, lib, args[m], n_launch if m == 'information_gain' else launches))
    med = {m: float(np.median(v)) for m, v in ms.items()}
    return med, ms, n_launch, terms_per_setting(e, lik, level)


def c3_arm(obe, method, cycles, warmup=3):
    import torch

    from oracle import obe_oracle as orc
    from oracle.scenarios import build_inputs, by_name
    sc = by_name('c3_pipulse')
    inp = build_inputs(sc, 1_000_000)
    eng = obe.OptBayesExpt('rabi', inp['setting_values'], inp['prior'], inp['cons'], scale=False,
                           likelihood_model='poisson', design_noise='likelihood', seed=3, utility_method=method)
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


STUDY_MODES = {'fixed': dict(design_noise='fixed'), 'likelihood': dict(design_noise='likelihood'),
               'information_gain': dict(design_noise='likelihood', utility_method='information_gain')}


def study_arm(obe, mode, seeds, steps, truth):
    """Median final posterior std of every parameter over `seeds` simulated Poisson experiments."""
    from oracle import obe_oracle as orc
    cons, n = (0.3,), 100_000
    a, b = truth[1], truth[2]
    s = (np.linspace(0.0, 6.0, 241),)
    model = obe.builtin('lorentzian_hwhm')
    stds = []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for seed in range(seeds):
            g = np.random.default_rng(100 + seed)
            prior = np.array([g.uniform(1.0, 5.0, n), g.uniform(0.25 * a, 2.0 * a, n), g.uniform(0.2 * b, 2.0 * b, n)])
            eng = obe.OptBayesExpt(model, s, prior, cons, likelihood_model='poisson', default_noise_std=5.0,
                                   seed=200 + seed, **STUDY_MODES[mode])
            eng.rng = np.random.default_rng(300 + seed)
            meas = np.random.default_rng(400 + seed)
            for _ in range(steps):
                x = eng.opt_setting()
                eng.pdf_update((x, float(meas.poisson(orc.model_lorentzian_hwhm(x, truth, cons)))))
            stds.append([float(v) for v in np.asarray(eng.std()).reshape(-1)[:3]])
    stds = np.array(stds)
    return np.median(stds, axis=0), stds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--cycles', type=int, default=300)
    ap.add_argument('--info-cycles', type=int, default=30)
    ap.add_argument('--seeds', type=int, default=16)
    ap.add_argument('--steps', type=int, default=150)
    ap.add_argument('--sizes', default='10000,100000')
    ap.add_argument('--skip', default='', help='comma-separated arms to skip: utility, c3, study')
    ap.add_argument('--out', default=os.path.join('profiles', 'information_gain_b200.jsonl'))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_information_gain.py measures on a CUDA device; none is visible')
    import optbayesexpt_b200 as obe
    name, power = card()
    base = dict(gpu=name, power_limit=power)
    skip = set(a.skip.split(','))
    lines = []

    def emit(d):
        lines.append(dict(base, **d))
        print(json.dumps(lines[-1]), flush=True)

    if 'utility' not in skip:
        arms = [('poisson', 1, 'broad'), ('poisson', 1, 'tight'), ('poisson', 100, 'broad'), ('poisson', 100, 'tight'),
                ('poisson', 10000, 'broad'), ('poisson', 10000, 'tight'), ('binomial', 10, 'broad'),
                ('binomial', 1000, 'broad')]
        for n_settings in (int(v) for v in a.sizes.split(',')):
            for lik, level, prior_kind in arms:
                med, ms, n_launch, terms = utility_arm(obe, torch, lik, level, prior_kind, n_settings, a.launches,
                                                       a.rounds)
                emit(dict(arm=f'utility_{lik}_{level}_{prior_kind}_{n_settings}', likelihood=lik, level=level,
                          prior=prior_kind, n_settings=n_settings, n_draws=30, terms_per_setting=round(terms, 1),
                          launches_variance=a.launches, launches_information_gain=n_launch, rounds=a.rounds,
                          variance_us=round(1e3 * med['variance'], 2),
                          information_gain_us=round(1e3 * med['information_gain'], 2),
                          ns_per_term=round(1e6 * med['information_gain'] / (terms * n_settings), 4),
                          information_gain_us_rounds=[round(1e3 * v, 2) for v in ms['information_gain']]))
    if 'c3' not in skip:
        rates = {'variance_approx': [], 'information_gain': []}
        fired = {'variance_approx': [], 'information_gain': []}
        for _ in range(2):
            for method in rates:
                r, f = c3_arm(obe, method, a.info_cycles if method == 'information_gain' else a.cycles)
                rates[method].append(round(r, 2))
                fired[method].append(f)
        for method in rates:
            emit(dict(arm=f'c3_{method}', model='rabi', likelihood='poisson', design_noise='likelihood',
                      utility_method=method, n=1_000_000, n_settings=101 * 101,
                      cycles=a.info_cycles if method == 'information_gain' else a.cycles, resamples=fired[method],
                      cycles_per_s_runs=rates[method], cycles_per_s=float(np.median(rates[method]))))
    if 'study' not in skip:
        for label, truth in (('original', (3.1, 40.0, 10.0)), ('low', (3.1, 4.0, 1.0))):
            res = {m: study_arm(obe, m, a.seeds, a.steps, truth) for m in STUDY_MODES}
            d = dict(arm=f'study_{label}', model='lorentzian_hwhm', likelihood='poisson', truth=list(truth),
                     n=100_000, n_settings=241, seeds=a.seeds, steps=a.steps, default_noise_std=5.0)
            for m, (med, stds) in res.items():
                d[f'median_std_{m}'] = [round(float(v), 5) for v in med]
                d[f'std_x0_{m}'] = [round(float(v), 5) for v in stds[:, 0]]
            emit(d)
    os.makedirs(os.path.dirname(a.out) or '.', exist_ok=True)
    with open(a.out, 'w') as f:
        for ln in lines:
            f.write(json.dumps(ln) + '\n')
    print('wrote', a.out)


if __name__ == '__main__':
    main()
