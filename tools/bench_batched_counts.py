"""Cost of the batched engines' count likelihoods (BatchedOptBayesExpt(..., likelihood_model=...)).

    python tools/bench_batched_counts.py [--instances 4096] [--particles 1e4] [--launches 50] [--cycles 100]
                                         [--rounds 3] [--seeds 1024] [--steps 150] [--out profiles/batched_counts_b200.jsonl]

Arms (one JSON line each, with the card's name and power limit read by nvidia-smi in the same run; the arms of one
comparison alternate `rounds` times in one process, CUDA events around `launches` back-to-back launches of the C entry,
median per-launch time):
  update_<model>        obe_batch_update (use_last, no resample) at instances x particles, the Gaussian handle against
                        the Poisson (lorentzian_hwhm) or binomial (lorentzian_dip) one, d = 3.
  select                obe_batch_select, 241 settings, K = 30, lorentzian_hwhm Poisson, 'fixed' against 'likelihood'.
  simulate_<arm>        obe_batch_simulate alone for `instances` instances at lambda ~ 1, 100, 1e4 and binomial n = 100.
  loop                  closed_loop_cycle, Gaussian against Poisson at instances x particles: cycles/s of wall time over
                        `cycles` cycles each, ending in a device synchronise.
  study                 DESIGN 6b's Poisson Lorentzian study (x0 = 3.1, a = 40, b = 10, hwhm 0.3, 241 settings, `steps`
                        measurements) as one batched engine of `seeds` seeds x 1e4 particles, 'fixed' (default_noise_std
                        = 5) against 'likelihood': median final std of (x0, a, b) and the wall time.
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

SETTINGS = np.linspace(1.5, 4.5, 241)


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power = (out[0].split(', ') + ['?'])[:2] if out else ('?', '?')
    return name, power


def prior(kind, g, B, n):
    if kind == 'peak':
        return np.stack([np.array([g.uniform(2.0, 4.0, n), g.uniform(20.0, 80.0, n), g.uniform(2.0, 20.0, n)])
                         for _ in range(B)])
    return np.stack([np.array([g.uniform(2.0, 4.0, n), g.uniform(0.2, 0.8, n), g.uniform(0.2, 0.6, n)])
                     for _ in range(B)])


def engine(kind, lik, B, n, **kw):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    g = np.random.default_rng(1)
    if kind == 'peak':
        return BatchedOptBayesExpt('lorentzian_hwhm', (SETTINGS,), prior('peak', g, B, n), (0.3,),
                                   likelihood_model=lik, seed=2, **kw)
    return BatchedOptBayesExpt('lorentzian_dip', (SETTINGS,), prior('dip', g, B, n), (), likelihood_model=lik, seed=2,
                               **kw)


def truths(kind, B):
    g = np.random.default_rng(3)
    if kind == 'peak':
        return np.stack([g.uniform(2.8, 3.4, B), np.full(B, 40.0), np.full(B, 10.0)], axis=1)
    return np.stack([g.uniform(2.8, 3.4, B), np.full(B, 0.5), np.full(B, 0.4)], axis=1)


def timed(torch, fn, launches):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches * 1e3          # us


def update_call(beng):
    from optbayesexpt_b200 import _lib
    lib = beng._lib

    def f():
        _lib.check(lib.obe_batch_update(beng._model, beng._bs(), C.c_void_p(beng._settings_dev.data_ptr()),
                                        beng._lds, 1, beng._cons_arr, None, beng.n_channels, 0, 0.0, -1.0, 0,
                                        beng._stream()))
    return f


def select_call(beng):
    return lambda: beng.opt_setting(sync=False)


def alternate(torch, calls, launches, rounds):
    """{arm: median us per launch} of the calls (name -> fn), alternated `rounds` times after one warm-up each."""
    for fn in calls.values():
        timed(torch, fn, 3)
    res = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            res[k].append(timed(torch, fn, launches))
    return {k: float(np.median(v)) for k, v in res.items()}, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--instances', type=int, default=4096)
    ap.add_argument('--particles', type=float, default=1e4)
    ap.add_argument('--launches', type=int, default=50)
    ap.add_argument('--cycles', type=int, default=100)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--seeds', type=int, default=1024)
    ap.add_argument('--steps', type=int, default=150)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'batched_counts_b200.jsonl'))
    args = ap.parse_args()
    import torch
    name, power = card()
    B, n = args.instances, int(args.particles)
    lines = []

    def emit(d):
        d.update(gpu=name, power_limit=power)
        print(json.dumps(d), flush=True)
        lines.append(d)

    warnings.simplefilter('ignore', RuntimeWarning)
    # ---- batched update: Gaussian against the count likelihoods
    for kind, lik, rec in (('peak', 'poisson', (3.0, 30.0, 0.0)), ('dip', 'binomial', (3.0, 60.0, 100.0))):
        engines = {'gaussian': engine(kind, None, B, n), lik: engine(kind, lik, B, n)}
        for e in engines.values():
            e.opt_setting(sync=False)
            e._record[:, 4] = rec[1]
            e._record[:, 8] = rec[2] if lik == 'binomial' else 1.0
        med, runs = alternate(torch, {k: update_call(e) for k, e in engines.items()}, args.launches, args.rounds)
        emit(dict(arm=f'update_{kind}', shape=[B, n, 3], us=med, runs_us=runs,
                  ratio=med[lik] / med['gaussian'], note='obe_batch_update, use_last, no resample test'))
        del engines
        torch.cuda.empty_cache()
    # ---- batched select: 'fixed' against 'likelihood'
    engines = {m: engine('peak', 'poisson', B, n, design_noise=m, default_noise_std=5.0) for m in ('fixed', 'likelihood')}
    med, runs = alternate(torch, {k: select_call(e) for k, e in engines.items()}, args.launches, args.rounds)
    emit(dict(arm='select', shape=[B, n, 241, 30], us=med, runs_us=runs, ratio=med['likelihood'] / med['fixed']))
    # ---- simulator kernel alone
    e = engines['fixed']
    res_sim = {}
    for lam in (1.0, 100.0, 1e4):
        tr = truths('peak', B)
        tr[:, 1], tr[:, 2] = 0.0, lam                    # lambda = b everywhere
        e.set_simulator(tr, seed=5)
        res_sim[f'poisson_{lam:g}'] = alternate(torch, {'x': lambda: e.simulate_measurement()}, args.launches,
                                                args.rounds)[0]['x']
    eb = engine('dip', 'binomial', B, 64, design_noise='likelihood', design_aux=100)
    eb.set_simulator(truths('dip', B), trials=100, seed=5)
    res_sim['binomial_100'] = alternate(torch, {'x': lambda: eb.simulate_measurement()}, args.launches,
                                        args.rounds)[0]['x']
    emit(dict(arm='simulate', instances=B, us=res_sim))
    del engines, e, eb
    torch.cuda.empty_cache()
    # ---- closed loop, Gaussian against Poisson
    loops = {}
    for lik in ('gaussian', 'poisson'):
        le = engine('peak', None if lik == 'gaussian' else 'poisson', B, n, default_noise_std=5.0,
                    design_noise='fixed')
        if lik == 'gaussian':
            le.set_simulator(truths('peak', B), 5.0, seed=7)
        else:
            le.set_simulator(truths('peak', B), seed=7)
        loops[lik] = le
    rates = {k: [] for k in loops}
    for k, le in loops.items():
        for _ in range(5):
            le.closed_loop_cycle()
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        for k, le in loops.items():
            t0 = time.perf_counter()
            for _ in range(args.cycles):
                le.closed_loop_cycle()
            torch.cuda.synchronize()
            rates[k].append(args.cycles / (time.perf_counter() - t0))
    med = {k: float(np.median(v)) for k, v in rates.items()}
    emit(dict(arm='loop', shape=[B, n, 241, 30], cycles_per_s=med, runs=rates,
              simulate_share_of_cycle={k: res_sim[k] * 1e-6 * med['poisson'] for k in res_sim}))
    del loops
    torch.cuda.empty_cache()
    # ---- the Poisson Lorentzian design study, `seeds` seeds in one batched engine
    S = args.seeds
    study = {}
    for mode in ('fixed', 'likelihood'):
        from optbayesexpt_b200.batched import BatchedOptBayesExpt
        g = np.random.default_rng(11)
        se = BatchedOptBayesExpt('lorentzian_hwhm', (SETTINGS,), prior('peak', g, S, 10000), (0.3,),
                                 likelihood_model='poisson', design_noise=mode, default_noise_std=5.0, seed=12)
        se.set_simulator(np.array([3.1, 40.0, 10.0]), seed=13)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            se.closed_loop_cycle()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        std = se.std()
        study[mode] = dict(median_std=np.median(std, axis=0).tolist(), wall_s=wall)
        del se
        torch.cuda.empty_cache()
    emit(dict(arm='study', seeds=S, particles=10000, steps=args.steps, truth=[3.1, 40.0, 10.0], hwhm=0.3, **study,
              x0_fixed_over_likelihood=study['fixed']['median_std'][0] / study['likelihood']['median_std'][0]))
    if args.out:
        with open(args.out, 'w') as f:
            for d in lines:
                f.write(json.dumps(d) + '\n')


if __name__ == '__main__':
    main()
