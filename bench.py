#!/usr/bin/env python
"""bench.py -- full pdf_update + resample + opt_setting cycles per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c1|c2|c3|c5|sweeper]
                    [--dump-outputs DIR]

Default workload c4 (BASELINE.json configs[3], fits one B200): synthetic Lorentzian cloud, 1e8 particles x
3 parameters, 1e5 settings, n_draws = 30, resample forced every cycle (resample_threshold > 1).
c1 / c2 / c3 are the reference's own demo shapes with their real models (Lorentzian / line + unknown sigma /
Rabi on the 101 x 101 grid), c5 the 4096 batched lock-in engines.  A "step" is one full cycle.  ONE JSON line.

  value      cycles/s with everything resident in HBM, no host synchronisation inside the timed
             region (run_cycle_async), CUDA events, max over ranks
  e2e        the same cycle through the reference-shaped API (pdf_update(record) -> opt_setting()),
             closed loop: the record goes host->device every step, the stats block and the chosen
             index come back every step
  roofline   dominant kernel (the one-kernel systematic resample) against the measured HBM peak
  cpu_baseline / --impl reference: the UNMODIFIED reference (baseline/_ref, see baseline/reference_arm.py)
             timed on the host: c1-c3 at their full size; c4 measured at 1e6 and 1e7 particles and extrapolated
             to 1e8 with the fitted exponent (labelled).  Falls back to the numpy port (oracle/) only when the
             reference is not installed.
  --dump-outputs DIR   (one GPU) after the timed steps, what the timed path handed its caller in its last step, as
             DIR/<name>.npy in float64, 64 MB at most: c1-c4 the chosen setting, the utility of every setting and the
             particles and weights at a fixed, seeded sample of at most 2^20 particles; c5 every instance's choice and
             moments and the clouds of 8 fixed instances; sweeper the posterior moments and a sample of the cloud.
             The inputs depend on the arguments only, so two builds run with the same arguments can be compared output
             for output.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

TRUE_PARS = (3.14, -1200.0, 50400.0)
SIGMA = 500.0
SETTLE_S = 0.5          # idle before each headline measurement of the c4 cycle (see settle() in main)
CONS = (0.1,)


def lorentz(x, p):
    return p[2] + p[1] / (((x - p[0]) / CONS[0]) ** 2 + 1)


def measured_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)         # (a no-op once stopped; ends the sampler if the run fails)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'),
                                     r[5:9]):
                    if val.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


DUMP_BYTES = 64 << 20        # --dump-outputs writes at most this much in all
DUMP_ROW = 1 << 20           # entries of the longest dumped row; a longer one is sampled


def _sample(n, m=DUMP_ROW):
    """A fixed, seeded, sorted sample of m of the indices 0..n-1 (all of them when n <= m)."""
    return np.arange(n) if n <= m else np.sort(np.random.default_rng(0).choice(n, m, replace=False))


def _cloud_sample(eng, max_bytes):
    """The cloud's particles and normalised weights at a fixed sample of the particle indices, within max_bytes.
    Both are gathered on the device, and nothing of the engine's state changes (the measurements after a dump see the
    engine the timed steps left)."""
    import ctypes
    import torch
    particles = eng.particles_dev                       # (waits for an enqueued cycle)
    m = int(min(DUMP_ROW, max_bytes // (8 * (eng.n_dims + 1))))
    idx = torch.from_numpy(_sample(eng.n_particles, m)).to(particles.device)
    w = torch.empty(eng.n_particles, dtype=torch.float64, device=particles.device)
    eng._check(eng._lib.obe_normalized_weights(eng._cs(), ctypes.c_void_p(w.data_ptr()), eng._stream()))
    return {'particles': particles[:, idx].cpu().numpy(), 'weights': w[idx].cpu().numpy()}


def _write_dump(out_dir, arrays):
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise RuntimeError(f'--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte budget')
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def dump_cycle(eng, out_dir):
    """--dump-outputs of an OptBayesExpt cycle (c1-c4): the chosen setting and its utility, the utility of every setting
    (a fixed sample of DUMP_ROW settings when there are more) and a sample of the resampled cloud."""
    import torch
    best = eng.best_index_dev.cpu()
    index = int(best[0])
    utility = eng._utility_dev
    out = {'chosen_index': [index], 'chosen_utility': best[1:2].view(torch.float64).numpy(),
           'chosen_setting': eng.allsettings[:, index]}
    if utility.numel() > DUMP_ROW:
        cols = _sample(utility.numel())
        out['utility_index'] = cols
        utility = utility[torch.from_numpy(cols).to(utility.device)]
    out['utility'] = utility.cpu().numpy()
    out.update(_cloud_sample(eng, DUMP_BYTES - sum(8 * np.size(a) for a in out.values())))
    _write_dump(out_dir, out)


def dump_batched(eng, out_dir, n_instances=8):
    """--dump-outputs of the batched cycle (c5): every instance's chosen setting, resample flag and posterior moments,
    and the whole clouds of a fixed sample of instances."""
    idx = eng.last_setting_index
    inst = _sample(eng.n_instances, n_instances)
    _write_dump(out_dir, {'chosen_index': idx, 'chosen_setting': eng.allsettings[:, idx],
                          'just_resampled': eng.just_resampled, 'mean': eng.mean(), 'covariance': eng.covariance(),
                          'n_eff': eng.n_eff(), 'instances': inst,
                          'particles': np.stack([eng.particles(b) for b in inst]),
                          'weights': np.stack([eng.particle_weights(b) for b in inst])})


# -------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference (baseline/reference_arm.py); the numpy port only as a fallback
# -------------------------------------------------------------------------------------------------
def port_cycle_rate(n_full, n_settings, n_draws, n_sample=1_000_000, budget_s=20.0, max_cycles=8):
    """Fallback when baseline/_ref is missing: the numpy restatement of the reference (oracle/), bounded sample,
    O(N) part scaled linearly.  kind = "port"."""
    from oracle import obe_oracle as orc
    rng = np.random.default_rng(1001)
    prior = np.array([rng.uniform(2, 4, n_sample), rng.uniform(-2000, -400, n_sample),
                      rng.normal(50000, 1000, n_sample)])
    settings = (np.linspace(1.5, 4.5, n_settings),)
    eng = orc.OracleOBE(orc.model_lorentzian_hwhm, settings, prior, CONS, n_draws=n_draws, scale=False,
                        default_noise_std=SIGMA, resample_threshold=2.0, rng=np.random.default_rng(1003))
    meas = np.random.default_rng(1002)
    t_n, t_grid, cycles = 0.0, 0.0, 0
    t_start = time.perf_counter()
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        while cycles < max_cycles and (time.perf_counter() - t_start) < budget_s:
            t0 = time.perf_counter()
            draws, _ = orc.randdraw(eng.particles, eng.particle_weights, eng.rng.random(n_draws))
            t1 = time.perf_counter()
            var_p, _ = orc.yvar_from_draws(eng.model, eng.allsettings, draws, CONS, 1)
            util = orc.utility_variance(var_p, orc.noise_var_default(SIGMA, 1))
            best = orc.opt_index(util)
            t2 = time.perf_counter()
            x = (eng.allsettings[0, best],)
            y = float(lorentz(x[0], TRUE_PARS) + SIGMA * meas.standard_normal())
            t3 = time.perf_counter()
            eng.pdf_update((x, y, SIGMA))          # update + forced multinomial resample
            t4 = time.perf_counter()
            t_n += (t1 - t0) + (t4 - t3)
            t_grid += (t2 - t1)
            cycles += 1
    per_cycle_sample = (t_n + t_grid) / cycles
    per_cycle_full = (t_n / cycles) * (n_full / n_sample) + t_grid / cycles
    return {
        'value': 1.0 / per_cycle_full, 'unit': 'cycles/s', 'cores': 1, 'kind': 'port',
        'sample': (f'FALLBACK (baseline/_ref missing): numpy port of the reference (oracle/) on {n_sample} particles x '
                   f'{n_settings} settings, {cycles} full cycles, {per_cycle_sample * 1e3:.1f} ms/cycle measured; O(N) part '
                   f'scaled x{n_full / n_sample:g} linearly'),
        'measured': [dict(n=n_sample, cycles=cycles, s_per_cycle=per_cycle_sample)], 'extrapolated': True,
        'ms_per_cycle': per_cycle_full * 1e3, 'timed_s': per_cycle_sample * cycles,
    }


def cpu_arm(workload, args, warmup, steps, budget_s, forced=True):
    """cpu_baseline object: the unmodified reference when it is installed (kind "reference"), else the port (c4)."""
    from baseline import reference_arm as ra
    out = ra.reference_rate(workload, forced=forced, warmup=warmup, steps=steps, budget_s=budget_s,
                            n_draws=args.draws, settings=args.settings)
    if 'unavailable' in out and workload == 'c4':
        why = out['unavailable']
        out = port_cycle_rate(int(args.particles), args.settings, args.draws, max_cycles=max(1, min(steps, 8)))
        out['reference_unavailable'] = why
    return out


def workload_config(workload, args):
    from baseline import reference_arm as ra
    wl = ra.WORKLOADS[workload]
    n_set = int(np.prod([len(v) for v in wl['settings']()])) if workload != 'c4' else args.settings
    n = wl['n_particles'] if workload != 'c4' else int(args.particles)
    d = len(wl['prior'](np.random.default_rng(0), 2))
    return {'workload': f'{wl["label"]} (BASELINE configs[{wl["config_index"]}])' if workload != 'c4' else
            f'synthetic Lorentzian scale-out: {n:.0e} particles x {n_set} settings, n_draws={args.draws}, d=3, '
            f'resample forced every cycle (BASELINE configs[3])',
            'particles': n, 'settings': n_set, 'n_draws': args.draws, 'n_params': d}


def reference_line(args):
    """--impl reference: the unmodified reference on the host cores, this arm's config/metric/unit.
    Each timed step is one closed-loop cycle of the reference on a bounded sample of the workload (c4: 1e6
    particles, then 2 cycles at 1e7 for the scaling exponent; c1-c3: the full workload); `value` is the rate at the
    workload's full size, `ms_per_step` what a step actually took."""
    wl = args.workload if args.workload in ('c1', 'c2', 'c3', 'c4') else 'c4'
    base = cpu_arm(wl, args, warmup=max(1, args.warmup), steps=max(1, args.steps), budget_s=240.0)
    if 'unavailable' in base:
        print(json.dumps({'impl': 'reference', 'unavailable': base['unavailable']}))
        return
    first = base['measured'][0]
    config = workload_config(wl, args)
    config['l2'] = 'n/a (host run)'
    line = {'impl': 'reference', 'metric': 'pdf_update+resample+opt_setting cycles/sec', 'value': base['value'],
            'unit': 'cycles/s', 'n_gpus': 0, 'steps': first['cycles'], 'warmup': max(1, args.warmup),
            'ms_per_step': first['s_per_cycle'] * 1e3,
            'ms_per_step_note': (f'a timed step is one reference cycle at {first["n"]:.0e} particles (what actually ran); '
                                 f'`value` is the rate at the full workload size'
                                 + (' (extrapolated, see cpu_baseline)' if base.get('extrapolated') else '')),
            'ms_per_cycle_full_workload': base['ms_per_cycle'],
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config, 'cpu_baseline': base,
            'e2e': {'value': base['value'], 'unit': 'cycles/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------
# c1 / c2 / c3: the reference's own demo shapes with their real models (one GPU)
# -------------------------------------------------------------------------------------------------
def bench_small(args):
    import torch
    import __graft_entry__
    __graft_entry__.build()
    import optbayesexpt_b200 as obe
    from baseline import reference_arm as ra
    wl = ra.WORKLOADS[args.workload]
    n = wl['n_particles']
    prior = wl['prior'](np.random.default_rng(1001), n)
    d = prior.shape[0]
    settings = wl['settings']()
    n_set = int(np.prod([len(v) for v in settings]))
    n_knobs = len(settings)

    def make(threshold):
        kw = dict(n_draws=args.draws, scale=False, seed=1003, resample_threshold=threshold)
        if wl['kind'] == 'noise':
            return obe.OptBayesExptNoiseParameter(wl['device_model'], settings, prior, wl['cons'],
                                                  noise_parameter_index=wl['noise_parameter_index'], **kw)
        return obe.OptBayesExpt(wl['device_model'], settings, prior, wl['cons'],
                                default_noise_std=wl['default_noise_std'], **kw)

    meas = np.random.default_rng(1002)
    import warnings
    warnings.simplefilter('ignore', RuntimeWarning)
    # ---- device-resident leg, resample forced every cycle, records prepared in advance, no host sync
    eng = make(2.0)
    xs = eng.allsettings
    recs = [ra.simulate(wl, tuple(xs[:, (7919 * t + n_set // 2) % n_set]), meas) for t in range(args.warmup + args.steps)]
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device='cuda')      # 256 MB > the 126 MB L2
    for t in range(max(args.warmup, 3)):
        eng.run_cycle_async(recs[t % len(recs)])
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for t in range(args.steps):
        flush.zero_()                                   # cold L2 for every timed cycle (outside the bracket)
        ev[t][0].record()
        eng.run_cycle_async(recs[args.warmup + t])
        ev[t][1].record()
    torch.cuda.synchronize()
    ms_cold = float(np.sum([a.elapsed_time(b) for a, b in ev])) / args.steps
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    for t in range(args.steps):
        eng.run_cycle_async(recs[args.warmup + t])
    b1.record()
    torch.cuda.synchronize()
    ms_warm = b0.elapsed_time(b1) / args.steps
    if args.dump_outputs:
        dump_cycle(eng, args.dump_outputs)

    # ---- end to end through pdf_update / opt_setting, closed loop: forced and natural resampling
    def closed_loop(threshold, steps):
        e = make(threshold)
        e.eager_select = True
        e.async_update = True            # (only takes effect where the resample decision is known: the forced loop)
        x = e.opt_setting()
        for _ in range(max(3, args.warmup)):
            e.pdf_update(ra.simulate(wl, x, meas))
            x = e.opt_setting()
        torch.cuda.synchronize()
        n_res = 0
        t0 = time.perf_counter()
        for _ in range(steps):
            e.pdf_update(ra.simulate(wl, x, meas))
            n_res += 1 if e.just_resampled else 0
            x = e.opt_setting()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps, n_res / steps
    e2e_steps = max(args.steps, 200 if n <= 100_000 else 50)
    s_forced, r_forced = closed_loop(2.0, e2e_steps)
    s_natural, r_natural = closed_loop(0.5, e2e_steps)
    clocks = sampler.stop()
    peak, peak_src = measured_peak()
    c_ch = 1
    b_cycle = 8.0 * n * (3 * d + 5 - 1) + 8.0 * n_set * (n_knobs + 1)      # SURVEY 8(d), offspring weights implicit
    config = workload_config(args.workload, args)
    config['l2'] = (f'working set {(8.0 * n * (2 * d + 2)) / 1e6:.1f} MB fits the 126 MB L2: `value` is measured with the L2 '
                    f'flushed (256 MB write) before every timed cycle, per-cycle CUDA events; `l2_resident` is the same '
                    f'loop back to back without the flush')
    config['resample'] = 'forced every cycle (value, e2e); natural rate in e2e_natural'
    line = {
        'metric': 'pdf_update+resample+opt_setting cycles/sec', 'value': 1e3 / ms_cold, 'unit': 'cycles/s', 'n_gpus': 1,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_cold, 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': config,
        'l2_resident': {'ms_per_step': ms_warm, 'cycles_per_s': 1e3 / ms_warm},
        'e2e': {'value': 1.0 / s_forced, 'unit': 'cycles/s', 'steps': e2e_steps, 'resamples_per_cycle': r_forced,
                'h2d_bytes_per_step': 8 * (n_knobs + 2 * c_ch + d + 1) + 8 * args.draws, 'd2h_bytes_per_step': 8 * 64 + 16,
                'note': 'record, pivot and uniforms travel as kernel arguments; stats block + argmax come back'},
        'e2e_natural': {'value': 1.0 / s_natural, 'unit': 'cycles/s', 'steps': e2e_steps,
                        'resamples_per_cycle': r_natural, 'resample_threshold': 0.5},
        'gpu_launches': 5 * args.steps + (args.steps if wl['kind'] == 'noise' else 0),
        'roofline': {'bound': 'hbm', 'kernel': 'whole cycle (update + plan + one-kernel resample + draw + utility)',
                     'achieved': b_cycle / (ms_cold * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                     'frac': b_cycle / (ms_cold * 1e-3) / 1e9 / peak, 'traffic': None,
                     'traffic_source': 'not captured for this shape (launch-latency-bound: 5 launches per cycle)',
                     'peak_source': peak_src, 'algorithmic_bytes_per_launch': b_cycle},
        'clocks': clocks,
    }
    if not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_arm(args.workload, args, warmup=2, steps=20 if n <= 100_000 else 8, budget_s=12.0)
        line['cpu_baseline_natural'] = cpu_arm(args.workload, args, warmup=2, steps=20 if n <= 100_000 else 8,
                                               budget_s=12.0, forced=False)
    print(json.dumps(line))


def lockin_model(w, pars):
    """(Re Z, Im Z) of R-L in parallel with C (demos/lockin/lockin_of_coil.py:63-102), for the simulated instrument."""
    L, R, Cc = pars[:3]
    z = 1 / (1 / (R + 1j * w * L) + 1j * w * Cc)
    return np.array((np.real(z), np.imag(z)))


# -------------------------------------------------------------------------------------------------
def bench_c5(args, rank, world):
    """BASELINE configs[4]: 4096 independent lock-in engines x 1e4 particles, batched; instances are split over
    the ranks with no collective at all (weak in nothing: the total is fixed -> strong scaling)."""
    import torch
    import torch.distributed as dist
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    B_total, n = 4096, 10000
    B = B_total // world
    g = torch.Generator(device='cuda')
    g.manual_seed(1001 + rank)
    prior = torch.empty((B, 4, n), dtype=torch.float64, device='cuda')
    for j, sc_ in enumerate((1e-3, 10.0, 1e-5, 10.0)):
        prior[:, j] = torch.empty((B, n), dtype=torch.float64, device='cuda').exponential_(1.0, generator=g) * sc_
    settings = (2 * np.pi * np.logspace(2, 6, 200),)
    eng = BatchedOptBayesExpt('lockin_coil', settings, prior, (), noise_parameter_index=(3, 3),
                              constraint_lt=(0, 1, 2, 3), cost_of_changing_setting=5.0, scale=False, seed=1003)
    del prior
    truth = (1.2e-3, 8.0, 0.9e-5)
    meas = np.random.default_rng(1002 + rank)

    def step(sync):
        out = eng.opt_setting(sync=sync)
        if sync:
            z = lockin_model(out[1][0], truth)
            y = z.T + 5.0 * meas.standard_normal((B, 2))
        else:
            y = step.y
        eng.pdf_update(y, force_resample=args.force_resample)
        step.y = y
    step.y = None
    # device-resident leg: the on-device MeasurementSimulator writes every instance's record (no H2D at all)
    eng.set_simulator(np.tile(np.array(truth), (B, 1)), 5.0, seed=1002 + rank)
    for _ in range(max(args.warmup, 3)):
        step(True)
    for _ in range(3):
        eng.closed_loop_cycle(force_resample=args.force_resample)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0.record()
    for _ in range(args.steps):
        eng.closed_loop_cycle(force_resample=args.force_resample)   # select -> simulate -> update/resample, no host
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_batched(eng, args.dump_outputs)
    # per-phase split of the same cycle (events between the phases; outside the timed region)
    pe = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    for t in range(args.steps):
        pe[t][0].record()
        eng.opt_setting(sync=False)
        pe[t][1].record()
        eng.simulate_measurement()
        pe[t][2].record()
        eng._update_from_record(1, eng.n_channels, args.force_resample)
        pe[t][3].record()
    torch.cuda.synchronize()
    split = [float(np.mean([pe[t][i].elapsed_time(pe[t][i + 1]) for t in range(args.steps)])) for i in range(3)]
    clocks = sampler.stop() if rank == 0 else None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(True)                        # e2e: chosen settings D2H, measurements H2D every cycle
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if world > 1:
        tt = torch.tensor([ms, e2e_s], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(tt[0]), float(tt[1])
        dist.destroy_process_group()
    if rank != 0:
        return
    peak, peak_src = measured_peak()
    d = 4
    b_cycle = 8.0 * n * B_total * ((d + 2) + (args.force_resample and (2 * d + 2) + (d + 1) or 0))
    line = {'metric': 'batched pdf_update+resample+opt_setting cycles/sec (4096 engines)', 'value': 1e3 / ms,
            'unit': 'batched cycles/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms,
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': 'batched demos/lockin: 4096 OBE instances x 1e4 particles, d=4, 2 channels, S=200 '
                                   '(BASELINE configs[4])', 'force_resample': bool(args.force_resample)},
            'instance_cycles_per_s': B_total * 1e3 / ms,
            'kernels_ms': {'select (draws + utility + argmax)': split[0], 'simulate measurement': split[1],
                           'update + resample of the flagged instances': split[2]},
            'gpu_launches': 6 * args.steps, 'clocks': clocks,
            'bound_note': 'update and select are barrier- and latency-bound (per-instance block barriers; FP64 pipe 35 % / '
                          '47 % busy): profiles/r2_ncu_summary.md, c5 section',
            'e2e': {'value': 1.0 / e2e_s, 'unit': 'batched cycles/s', 'h2d_bytes_per_step': B * 12 * 8,
                    'd2h_bytes_per_step': B * 8},
            'roofline': {'bound': 'hbm', 'achieved': b_cycle / world / (ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                         'frac': b_cycle / world / (ms * 1e-3) / 1e9 / peak, 'traffic': None, 'peak_source': peak_src,
                         'kernel': 'whole batched cycle (update + resample of flagged instances + select)'},
            'reference_note': 'one reference instance runs 488 cycles/s on one CPU core (BASELINE.md): 4096 instances '
                              '~ 8.4 s per batched cycle'}
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------
def bench_sweeper(args):
    """SURVEY 8(f) row 2: the sweeper's inference half.  One sweep = 64 measured points digested by
    OptBayesExptSweeper.pdf_update on 1e7 particles (d = 4, sigma unknown); fused multi-point kernel against the
    reference's loop of one update per point.  Resample test on (threshold 0.5), systematic resampling."""
    import torch
    import __graft_entry__
    __graft_entry__.build()
    import optbayesexpt_b200 as obe
    n, m = int(args.particles) if args.particles < 1e8 else 10_000_000, 64
    g = torch.Generator(device='cuda')
    g.manual_seed(1001)
    f64 = dict(dtype=torch.float64, device='cuda')
    xvals = np.linspace(1.5, 4.5, 1000)
    truth, noise = (3.2, 1500.0, 300.0), 300.0

    def make():
        prior = torch.empty((4, n), **f64)
        prior[0] = 2 + 2 * torch.rand(n, generator=g, **f64)
        prior[1] = 400 + 1600 * torch.rand(n, generator=g, **f64)
        prior[2] = 500 + 1000 * torch.randn(n, generator=g, **f64)
        prior[3] = torch.empty(n, **f64).exponential_(1.0, generator=g) * 500
        return obe.OptBayesExptSweeper('lorentzian_hwhm', (xvals,), prior, (0.1,), noise_parameter_index=3,
                                       scale=False, seed=7)
    out = {}
    for mode in ('fused', 'point_by_point'):
        g.manual_seed(1001)                       # same cloud, same sweeps, same noise for both modes
        meas = np.random.default_rng(1002)
        eng = make()
        eng.fused_sweep = (mode == 'fused')
        times, n_res = [], 0
        for it in range(args.warmup + args.steps):
            start = int(meas.integers(0, len(xvals) - m))
            xs = xvals[start:start + m]
            ys = lorentz(xs, truth) + noise * meas.standard_normal(m)
            e0 = eng._epoch
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.pdf_update(((xs,), ys))
            torch.cuda.synchronize()
            if it >= args.warmup:
                times.append(time.perf_counter() - t0)
                n_res += eng._epoch - e0
        out[mode] = (float(np.mean(times)), n_res / max(1, args.steps))
        if args.dump_outputs and mode == 'fused':
            # what the last timed sweep left: the posterior cloud (a sample of it) and its moments
            _write_dump(args.dump_outputs, {'mean': eng.mean(), 'covariance': eng.covariance(),
                                            **_cloud_sample(eng, DUMP_BYTES // 2)})
        del eng
        torch.cuda.empty_cache()
    t_f, r_f = out['fused']
    t_p, r_p = out['point_by_point']
    line = {'metric': 'sweeper pdf_update: measured points digested per second', 'value': m / t_f, 'unit': 'points/s',
            'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': t_f * 1e3, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': f'demos/sweeper inference half: {n:.0e} particles, d=4, sweeps of {m} points, '
                                   'resample test after every point (threshold 0.5)'},
            'point_by_point': {'value': m / t_p, 'unit': 'points/s', 'ms_per_sweep': t_p * 1e3,
                               'resamples_per_sweep': r_p},
            'resamples_per_sweep': r_f, 'speedup_vs_point_by_point': t_p / t_f,
            'e2e': {'value': m / t_f, 'unit': 'points/s', 'h2d_bytes_per_step': m * 96, 'd2h_bytes_per_step': 16},
            'note': 'wall clock around pdf_update incl. host synchronisation (the resample decisions are host-side)'}
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------
def invariance_check(world, rank, torch, obe):
    """SURVEY 8(e): the results must not depend on the number of GPUs.  A 1e6-particle side problem (outside every
    timed region): the cloud sharded over the `world` ranks against the single-cloud engine on the same GPU, same
    seeds -- chosen setting index identical; N_eff / mean to 1e-12 (the global sums are combined in rank order, a
    different association than one pass, so they agree to rounding, not to the bit); after a forced resample with
    the same comb offset and Philox stream every shard equals its slice of the single cloud's offspring (ancestors
    and jitter; tolerance 1e-12 relative + 1e-9 of the spread, the Cholesky factor inherits the rounding of the
    moments); shard lengths sum to n; the plan's overflow word is 0."""
    from optbayesexpt_b200 import _lib
    from optbayesexpt_b200.sharded import ShardedOptBayesExpt
    import warnings
    n, n_set = 1_000_000, 2000
    g = np.random.default_rng(4242)
    prior = np.array([g.uniform(2, 4, n), g.uniform(-2000, -400, n), g.normal(50000, 1000, n)])
    settings = (np.linspace(1.5, 4.5, n_set),)
    lo, hi = n * rank // world, n * (rank + 1) // world
    kw = dict(n_draws=30, scale=False, default_noise_std=SIGMA, seed=99)
    sh = ShardedOptBayesExpt('lorentzian_hwhm', settings, prior[:, lo:hi], CONS, **kw)
    one = obe.OptBayesExpt('lorentzian_hwhm', settings, prior, CONS, **kw)
    out = dict(n=n, cycles=3, chosen_index_equal=True, n_eff_rel=0.0, mean_rel=0.0, particles_err_in_tol_units=0.0,
               counts_sum_ok=True, overflow=0.0)
    meas = np.random.default_rng(700)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for e in (sh, one):
            e.tuning_parameters['auto_resample'] = False
        for t in range(out['cycles']):
            sh.rng, one.rng = np.random.default_rng(500 + t), np.random.default_rng(500 + t)
            xs, x1 = sh.opt_setting(), one.opt_setting()
            out['chosen_index_equal'] &= bool(sh.last_setting_index == one.last_setting_index and xs == x1)
            rec = (xs, float(lorentz(xs[0], TRUE_PARS) + SIGMA * meas.standard_normal()), SIGMA)
            sh.pdf_update(rec)
            one.pdf_update(rec)
            out['n_eff_rel'] = max(out['n_eff_rel'], abs(sh.n_eff() - one.n_eff()) / one.n_eff())
            out['mean_rel'] = max(out['mean_rel'], float(np.max(np.abs(sh.mean() - one.mean()) / np.abs(one.mean()))))
            sh._philox_seed = one._philox_seed = 4242 + t
            sh._epoch = one._epoch = t
            u0 = sh._u0                                    # the comb offset of the current shard plan
            saved, one.rng = one.rng, type('U0', (), {'random': staticmethod(lambda *a: u0)})()
            sh.resample()
            one.resample()
            one.rng = saved
            counts = sh.shard_counts
            out['counts_sum_ok'] &= bool(int(counts.sum()) == n)
            start = int(counts[:rank].sum())
            got = sh.particles
            want = one.particles[:, start:start + got.shape[1]]
            spread = want.std(axis=1, keepdims=True)
            err = np.abs(got - want) / (np.abs(want) * 1e-12 + spread * 1e-9)
            out['particles_err_in_tol_units'] = max(out['particles_err_in_tol_units'], float(err.max()))
            out['overflow'] = max(out['overflow'], float(sh._plan[_lib.PLAN_OVERFLOW].item()))
            out['shard_counts'] = [int(c) for c in counts]
    ok = (out['chosen_index_equal'] and out['n_eff_rel'] < 1e-12 and out['mean_rel'] < 1e-12
          and out['particles_err_in_tol_units'] <= 1.0 and out['counts_sum_ok'] and out['overflow'] == 0.0)
    import torch.distributed as dist
    flags = torch.tensor([1.0 if ok else 0.0, out['n_eff_rel'], out['mean_rel'], out['particles_err_in_tol_units']],
                         dtype=torch.float64, device='cuda')
    worst = flags.clone()
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    out['ok'] = bool(flags[0].item() > 0.5)
    out['n_eff_rel'], out['mean_rel'], out['particles_err_in_tol_units'] = [float(v) for v in worst[1:]]
    out['tolerances'] = {'chosen_index': 'identical', 'n_eff_rel': 1e-12, 'mean_rel': 1e-12,
                         'particles': '1e-12 relative + 1e-9 of the spread (1.0 = at tolerance)'}
    sh.close()
    return out


# -------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--particles', type=float, default=1e8)
    ap.add_argument('--settings', type=int, default=100000)
    ap.add_argument('--draws', type=int, default=30)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--force-resample', action='store_true')
    ap.add_argument('--workload', default='c4', choices=['c4', 'c1', 'c2', 'c3', 'c5', 'sweeper'],
                    help='c4: 1e8-particle Lorentzian cloud (default, the metric); c1/c2/c3: the reference demo shapes '
                         'with their real models (find_peak / line+noise / pipulse); c5: 4096 batched lock-in engines; '
                         'sweeper: the sweeper demo\'s multi-point inference (1 GPU)')
    ap.add_argument('--no-multinomial', action='store_true', help='c4: skip the like-for-like multinomial line')
    ap.add_argument('--no-invariance', action='store_true', help='multi-GPU: skip the G-invariance side check')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='one GPU: write the outputs of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    n_total = int(args.particles)
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.dump_outputs and (args.impl != 'ours' or world > 1):
        ap.error('--dump-outputs covers the GPU path on one GPU (--impl ours, no torchrun)')
    if args.impl == 'reference':
        return reference_line(args) if rank == 0 else None
    if args.workload == 'c5':
        return bench_c5(args, rank, world)
    if args.workload == 'sweeper':
        return bench_sweeper(args) if rank == 0 else None
    if args.workload in ('c1', 'c2', 'c3'):
        return bench_small(args) if rank == 0 else None      # replicas only: these shapes do not shard
    config = workload_config('c4', args)
    shard_mb = 8.0 * n_total * 4 / world / 1e6
    config['l2'] = (f'inputs ({shard_mb / 1e3:.2f} GB per GPU and cycle) are {shard_mb / 126:.1f}x the 126 MB L2 and every '
                    'cycle streams them once front to back: no flush needed'
                    if shard_mb > 2 * 126 else f'per-GPU working set {shard_mb:.0f} MB is within reach of the 126 MB L2: '
                    'L2-resident number, no flush')
    config['protocol'] = (f'value: {SETTLE_S} s idle, 3 warm-up cycles, K device-resident cycles (CUDA events); e2e: {SETTLE_S} s '
                          'idle, 3 warm-up cycles, K closed-loop cycles through pdf_update/opt_setting (host clock); '
                          'sustained: > 1 s back to back')

    import torch
    import torch.distributed as dist
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    import optbayesexpt_b200 as obe

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world > 1:
        from optbayesexpt_b200.sharded import ShardedOptBayesExpt
    n_local = n_total // world + (1 if rank < n_total % world else 0)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(1001 + rank)
    prior = torch.empty((3, n_local), dtype=torch.float64, device='cuda')
    prior[0] = 2 + 2 * torch.rand(n_local, generator=gen, dtype=torch.float64, device='cuda')
    prior[1] = -2000 + 1600 * torch.rand(n_local, generator=gen, dtype=torch.float64, device='cuda')
    prior[2] = 50000 + 1000 * torch.randn(n_local, generator=gen, dtype=torch.float64, device='cuda')
    settings = (np.linspace(1.5, 4.5, args.settings),)
    kw = dict(n_draws=args.draws, scale=False, default_noise_std=SIGMA, seed=1003, resample_threshold=2.0)
    if world > 1:
        eng = ShardedOptBayesExpt('lorentzian_hwhm', settings, prior, CONS, **kw)
    else:
        eng = obe.OptBayesExpt('lorentzian_hwhm', settings, prior, CONS, **kw)
    del prior
    meas = np.random.default_rng(1002)
    xs = settings[0]

    def record_for(x):
        return ((float(x),), float(lorentz(x, TRUE_PARS) + SIGMA * meas.standard_normal()), SIGMA)

    # ---------------- device-resident throughput: no host sync inside the timed region -----------
    fixed = [record_for(xs[(7919 * t + 50000) % len(xs)]) for t in range(args.warmup + args.steps)]
    for t in range(args.warmup):
        eng.run_cycle_async(fixed[t])
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    early = bool(eng._early_select_ok())
    e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def settle():
        """Both headline numbers (`value`, `e2e`) start from the same state: the cycle draws ~1 kW (FP64 + HBM) and
        the board's power cap pulls the SM clock down within ~0.1 s of sustained load, so each measurement is
        preceded by SETTLE_S of idle and its own warm-up cycles; `sustained` below is the long-run figure."""
        barrier()
        time.sleep(SETTLE_S)
        barrier()
    settle()
    for t in range(3):
        eng.run_cycle_async(fixed[t % len(fixed)])
    barrier()
    t_host0 = time.perf_counter()
    e_start.record()
    for t in range(args.steps):
        # the whole cycle, one C call (obe_cycle): update (+ stats exchange and shard plan when sharded) -> plan ->
        # [pick K draws, utility, argmax] || [streaming resample] -> join
        eng.run_cycle_async(fixed[args.warmup + t])
    e_stop.record()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / args.steps
    barrier()
    ms_total = e_start.elapsed_time(e_stop)
    if args.dump_outputs:
        dump_cycle(eng, args.dump_outputs)
    # ---------------- end to end through the reference-shaped API, closed loop -------------------
    eng.eager_select = True              # the resample inside pdf_update starts the selection opt_setting() asks for
    eng.async_update = True              # forced resampling: the decision does not need N_eff, pdf_update does not sync
    x = eng.opt_setting()
    for _ in range(max(3, args.warmup // 2)):
        eng.pdf_update(record_for(x[0]))
        x = eng.opt_setting()
    settle()
    for _ in range(3):
        eng.pdf_update(record_for(x[0]))
        x = eng.opt_setting()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        eng.pdf_update(record_for(x[0]))     # H2D: the record; D2H: the stats block (N_eff decision)
        x = eng.opt_setting()                # H2D: 30 uniforms; D2H: the chosen index
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([e2e_s], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    # the same closed loop at the NATURAL resample rate (threshold 0.5): the resample test runs on the device, most cycles
    # are update + selection only (single GPU; a sharded cloud decides on the host from the combined stats)
    e2e_natural = None
    if world == 1:
        eng.tuning_parameters['resample_threshold'] = 0.5
        for _ in range(5):
            eng.pdf_update(record_for(x[0]))
            x = eng.opt_setting()
        settle()
        for _ in range(3):
            eng.pdf_update(record_for(x[0]))
            x = eng.opt_setting()
        torch.cuda.synchronize()
        n_res, t0 = 0, time.perf_counter()
        for _ in range(e2e_steps):
            eng.pdf_update(record_for(x[0]))
            x = eng.opt_setting()
            n_res += 1 if eng.just_resampled else 0
        torch.cuda.synchronize()
        e2e_natural = {'value': e2e_steps / (time.perf_counter() - t0), 'unit': 'cycles/s', 'steps': e2e_steps,
                       'resamples_per_cycle': n_res / e2e_steps, 'resample_threshold': 0.5,
                       'device_resample_test': bool(eng._pending_cycle is not None and eng._device_test_ok())}
        eng.tuning_parameters['resample_threshold'] = 2.0
        eng.pdf_update(record_for(x[0]))            # back to a freshly resampled cloud for the diagnostics below
        x = eng.opt_setting()
    eng.eager_select = eng.async_update = False
    # the same cycle once more with an event between the update and the rest (per-phase split of the overlapped cycle)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    for t in range(args.steps):
        rec = fixed[args.warmup + t]
        ev[t][0].record()
        eng.run_cycle_async(rec, resample=False, select=False)     # update (+ stats exchange and shard plan when sharded)
        ev[t][1].record()
        eng.resample_select_async()
        ev[t][2].record()
    barrier()
    t_upd = float(np.mean([ev[t][0].elapsed_time(ev[t][1]) for t in range(args.steps)]))
    t_res = float(np.mean([ev[t][1].elapsed_time(ev[t][2]) for t in range(args.steps)]))
    # the same cycle with the selection serialised after the resample (early select off): the per-phase split
    eng.early_select = False
    sv = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.steps)]
    for t in range(2):
        eng.run_cycle_async(fixed[t % len(fixed)])
    barrier()
    s_start, s_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s_start.record()
    for t in range(args.steps):
        rec = fixed[args.warmup + t]
        sv[t][0].record()
        if world > 1:                    # the update kernel alone, then the stats exchange + shard plan
            obe.OptBayesExpt.run_cycle_async(eng, rec, resample=False, select=False)
            sv[t][4].record()
            eng._make_plan()
        else:
            eng.run_cycle_async(rec, resample=False, select=False)
            sv[t][4].record()
        sv[t][1].record()
        eng.resample_select_async(True, False)
        sv[t][2].record()
        eng.resample_select_async(False, True)
        sv[t][3].record()
    s_stop.record()
    barrier()
    eng.early_select = True
    ser = [float(np.mean([sv[t][i].elapsed_time(sv[t][i + 1]) for t in range(args.steps)])) for i in range(3)]
    ser.append(s_start.elapsed_time(s_stop) / args.steps)
    ser.append(float(np.mean([sv[t][4].elapsed_time(sv[t][1]) for t in range(args.steps)])))   # exchange + shard plan
    if world > 1:
        tt = torch.tensor([ms_total, t_upd, t_res] + ser, dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        vals = [float(v) for v in tt.cpu()]
        ms_total, t_upd, t_res, ser = vals[0], vals[1], vals[2], vals[3:]
    ms_step = ms_total / args.steps

    # ---------------- the cycle without a resample (SURVEY 8d: cycle_noresample) ------------------
    # update + select only; the weight row is explicit here, so the update moves 8N(d+2) bytes.  Single GPU
    # only (the sharded plan kernel would need a no-op resample to keep the ranks in step).
    ms_nores = None
    if world == 1:
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for t in range(3):
            eng.run_cycle_async(fixed[t % len(fixed)], resample=False, select=True)
        n0.record()
        for t in range(args.steps):
            eng.run_cycle_async(fixed[args.warmup + t], resample=False, select=True)
        n1.record()
        torch.cuda.synchronize()
        ms_nores = n0.elapsed_time(n1) / args.steps
        eng.resample()                       # back to a healthy cloud for the closed loop below

    # ---------------- the long-run figure: > 1 s of back-to-back cycles (the power cap has bitten by then) ----------
    n_sus = int(min(2000, max(50, 1.2 / (ms_step * 1e-3))))
    for t in range(3):
        eng.run_cycle_async(fixed[t % len(fixed)])
    barrier()
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u0.record()
    for t in range(n_sus):
        eng.run_cycle_async(fixed[t % len(fixed)])
    u1.record()
    barrier()
    ms_sus = u0.elapsed_time(u1) / n_sus
    if world > 1:
        tt = torch.tensor([ms_sus], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_sus = float(tt.item())
    clocks = sampler.stop() if rank == 0 else None

    # ---------------- outside every timed region: sanity of the sharded run, G-invariance side problem --------
    invariance = None
    if world > 1:
        from optbayesexpt_b200 import _lib as _obe_lib
        counts = eng.shard_counts
        assert int(counts.sum()) == n_total, f'shard lengths {counts} do not sum to {n_total}'
        eng._fetch_plan()
        assert float(eng._plan[_obe_lib.PLAN_OVERFLOW].item()) == 0.0, 'a shard overflowed its capacity / exchange timed out'
        if not args.no_invariance:
            invariance = invariance_check(world, rank, torch, obe)
            invariance['bench_shard_counts'] = [int(c) for c in counts]

    # ---------------- like for like: the reference's multinomial algorithm on the device (N = 1) --------------
    multinomial = None
    if world == 1 and not args.no_multinomial:
        eng.resampling = 'multinomial_device'
        k_m = max(3, min(10, args.steps))
        for t in range(2):
            eng.run_cycle_async(fixed[t % len(fixed)])
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for t in range(k_m):
            eng.run_cycle_async(fixed[t % len(fixed)])
        m1.record()
        torch.cuda.synchronize()
        ms_m = m0.elapsed_time(m1) / k_m
        multinomial = {'ms_per_step': ms_m, 'cycles_per_s': 1e3 / ms_m, 'steps': k_m,
                       'note': 'same ALGORITHM as the reference (N i.i.d. uniforms -> CDF -> searchsorted -> gather -> '
                               'Liu-West), all on the device: k_cdf + k_search + k_gather_jitter, uniforms from torch\'s CUDA '
                               'generator, Philox normals; the systematic comb above is the default fast path'}
        eng.resampling = 'systematic'

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peak()
    d = 3
    # The resample is forced every cycle, so the update always finds the offspring's implicit uniform weights
    # (never stored, never read): it moves d particle rows in and one weight row out, 8N(d+1), not the 8N(d+2)
    # of an update that follows an update.
    b_upd = 8.0 * n_total * (d + 1)
    b_res = 8.0 * n_total * (2 * d + 2)                # SURVEY 8(d): read w, gather d rows, write d rows, write w
    b_res_moved = 8.0 * n_total * (2 * d + 1)          # what this build has to move: the offspring weights stay implicit
    b_sel = 8.0 * args.settings * 2
    b_cycle = b_upd + b_res + b_sel
    gbs_res = b_res / world / (t_res * 1e-3) / 1e9
    fused = os.environ.get('OBE_OPT_RESAMPLE_FUSED', '1') != '0'
    sharded_launches = 0 if world == 1 else (2 if getattr(eng, '_peer', None) is not None else 1)
    line = {
        'metric': 'pdf_update+resample+opt_setting cycles/sec', 'value': 1e3 / ms_step, 'unit': 'cycles/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': config,
        'e2e': {'value': e2e_steps / e2e_s, 'unit': 'cycles/s',
                'h2d_bytes_per_step': 8 * (1 + 1 + 1 + 8 + 1) + 8 * args.draws,
                'd2h_bytes_per_step': 8 * 64 + 16,
                'note': 'record, pivot and uniforms travel as kernel arguments; stats block + argmax come back'},
        # update, plan, pick (the K draws, from the plan), utility, streaming resample (two kernels on the ancestors +
        # move path, which also draws with k_draw); sharded: + shard plan (peer exchange fused in) + draw collect
        'gpu_launches': ((5 if fused else 6) + sharded_launches) * args.steps,
        'roofline': {'bound': 'hbm',
                     'kernel': ('resample step = k_sys_plan + k_sys_resample_warp (one event bracket; the K-draw pick, '
                                'utility and argmax kernels run inside the same bracket on the selection stream)' if fused
                                else 'resample step = k_sys_plan + k_sys_ancestors + k_sys_move (one event bracket)'),
                     'achieved': gbs_res, 'peak': peak, 'unit': 'GB/s', 'frac': gbs_res / peak,
                     'algorithmic_bytes_per_launch': b_res / world,
                     'algorithmic_note': 'SURVEY 8(d): 8N(2d+2) (read w, gather d rows, write d rows, write w)',
                     'moved_bytes_per_launch': b_res_moved / world,
                     'frac_of_moved_bytes': b_res_moved / world / (t_res * 1e-3) / 1e9 / peak,
                     # dram__bytes_read.sum + dram__bytes_write.sum of the resample kernels from the ncu --set full capture
                     # of this build (profiles/r2_ncu_summary.md): bytes per particle at d = 3, scaled to this launch
                     'traffic': (56.3 if fused else 63.8) * n_total / world if d == 3 else None,
                     'traffic_source': 'profiles/r2_ncu_summary.md (ncu --set full of the same build and workload; '
                                       'per-particle figure x particles of this launch, not re-measured in this run)',
                     'peak_source': peak_src},
        'kernels_ms': {'update': t_upd, 'resample || draw+utility+argmax': t_res},
        'early_select': early, 'host_enqueue_ms_per_step': host_enqueue_ms,
        'serialised_cycle': {'note': 'same cycle, selection AFTER the resample on one stream (early select off)',
                             'ms_per_step': ser[3],
                             'kernels_ms': {'update': ser[0], 'resample': ser[1], 'draw+utility+argmax': ser[2]},
                             'stats_exchange_and_shard_plan_ms': ser[4] if world > 1 else None},
        'kernels_gbs': {'update': b_upd / world / (t_upd * 1e-3) / 1e9, 'resample': gbs_res},
        'exchange': None if world == 1 else ('peer (CUDA IPC over NVLink)' if getattr(eng, '_peer', None) is not None
                                             else 'nccl'),
        'cycle_hbm_frac': b_cycle / world / (ms_step * 1e-3) / 1e9 / peak,
        'cycle_noresample': None if ms_nores is None else {
            'ms_per_step': ms_nores, 'cycles_per_s': 1e3 / ms_nores,
            'hbm_frac': (8.0 * n_total * (d + 2) + b_sel) / (ms_nores * 1e-3) / 1e9 / peak},
        'sustained': {'cycles_per_s': 1e3 / ms_sus, 'ms_per_step': ms_sus, 'steps': n_sus,
                      'note': 'the same device-resident cycle back to back for > 1 s: the long-run rate under the board '
                              'power cap (`value` and `e2e` are K-cycle measurements, each after %.1f s of idle and '
                              'its own warm-up cycles)' % SETTLE_S},
        'clocks': clocks,
    }
    if e2e_natural is not None:
        line['e2e_natural'] = e2e_natural
    if multinomial is not None:
        line['multinomial_device'] = multinomial
    if invariance is not None:
        line['invariance'] = invariance
    try:
        fp = json.load(open(os.path.join(ROOT, 'profiles', 'fp64_peak.json')))
        line['fp64_peak_tflops'] = fp.get('fp64_tflops')
    except Exception:
        pass
    if not args.no_cpu_baseline and world == 1:       # the CPU arm is timed at N = 1 only
        line['cpu_baseline'] = cpu_arm('c4', args, warmup=1, steps=5, budget_s=30.0)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
