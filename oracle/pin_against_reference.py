"""Pin the oracle against the UNMODIFIED reference and write tests/golden/*.npz.

TEST INFRASTRUCTURE.  Needs a source tree of the reference (usnistgov/optbayesexpt
v1.2.0, given with --reference); the tests only read what it writes.  It imports
the reference from a scratch copy (numba writes a cache next to the source it
imports), seeds the reference's instance Generator (``obe.rng``, particlepdf.py:142-145) and runs each scenario
in lock-step with ``oracle.obe_oracle.OracleOBE`` seeded identically.  Every
step must agree (indices exactly, floats to 1e-12) or the script exits non-zero;
the reference's own trajectory is what gets written to tests/golden/.

    python oracle/pin_against_reference.py --reference SRC            # check + (re)write goldens
    python oracle/pin_against_reference.py --reference SRC --check    # check only

What is written is cut down by shrink() so that every golden file stays well under 1 MB.
"""
import argparse
import os
import shutil
import sys
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import obe_oracle as orc  # noqa: E402
from oracle.scenarios import SCENARIOS, build_inputs, simulate_measurement  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def import_reference(src):
    if not os.path.isdir(os.path.join(src, 'optbayesexpt')):
        raise SystemExit(f'no reference source tree at {src}')
    scratch = os.path.join(tempfile.gettempdir(), 'obe_refcopy')
    if os.path.isdir(scratch):
        shutil.rmtree(scratch)
    shutil.copytree(src, scratch)
    os.environ.setdefault('NUMBA_CACHE_DIR', os.path.join(tempfile.gettempdir(), 'numba_cache'))
    sys.dont_write_bytecode = True
    sys.path.insert(0, scratch)
    warnings.simplefilter('ignore', SyntaxWarning)
    import optbayesexpt  # noqa
    return optbayesexpt


def make_reference_engine(ref, sc, inp):
    model = orc.MODELS[sc['model']][0]
    kw = dict(n_draws=sc['n_draws'], scale=sc['scale'], a_param=sc['a_param'],
              resample_threshold=sc['resample_threshold'])
    if sc.get('choke') is not None:
        kw['choke'] = sc['choke']
    if sc['kind'] == 'base':
        obe = ref.OptBayesExpt(model, inp['setting_values'], inp['prior'], inp['cons'],
                               default_noise_std=sc.get('default_noise_std', 1.0), **kw)
    elif sc['kind'] == 'noise':
        obe = ref.OptBayesExptNoiseParameter(model, inp['setting_values'], inp['prior'], inp['cons'],
                                             noise_parameter_index=sc['noise_parameter_index'], **kw)
    elif sc['kind'] == 'lockin':
        # the subclass of demos/lockin/lockin_of_coil.py:107-153, re-stated through the
        # reference's own override protocol (the demo file itself imports matplotlib)
        class LockinClean(ref.OptBayesExptNoiseParameter):
            def __init__(self, *a, cost_of_changing_setting=1.0, **k):
                ref.OptBayesExptNoiseParameter.__init__(self, *a, **k)
                self.cost_of_changing_setting = cost_of_changing_setting

            def enforce_parameter_constraints(self):
                self.particle_weights = orc.enforce_all_nonnegative(self.parameters, self.particle_weights)

            def cost_estimate(self):
                return orc.lockin_cost(self.allsettings.shape[1], self.last_setting_index,
                                       self.cost_of_changing_setting)
        obe = LockinClean(model, inp['setting_values'], inp['prior'], inp['cons'],
                          noise_parameter_index=sc['noise_parameter_index'],
                          cost_of_changing_setting=sc['cost_of_changing_setting'], **kw)
    else:
        raise ValueError(sc['kind'])
    obe.rng = np.random.default_rng(sc['seed_rng'])
    return obe


def make_oracle_engine(sc, inp):
    model, _, _, _, nch = orc.MODELS[sc['model']]
    return orc.OracleOBE(
        model, inp['setting_values'], inp['prior'], inp['cons'], n_channels=nch,
        n_draws=sc['n_draws'], choke=sc.get('choke'), pickiness=sc.get('pickiness', 15),
        default_noise_std=sc.get('default_noise_std', 1.0), a_param=sc['a_param'],
        resample_threshold=sc['resample_threshold'], scale=sc['scale'],
        noise_parameter_index=sc.get('noise_parameter_index'),
        nonneg_constraint=(sc['kind'] == 'lockin'),
        cost_of_changing_setting=sc.get('cost_of_changing_setting'),
        rng=np.random.default_rng(sc['seed_rng']))


def run_lockstep(ref, sc):
    inp = build_inputs(sc)
    robe = make_reference_engine(ref, sc, inp)
    oobe = make_oracle_engine(sc, inp)
    meas_rng = np.random.default_rng(sc['seed_meas'])
    model = orc.MODELS[sc['model']][0]
    nch = orc.MODELS[sc['model']][4]
    T = sc['n_cycles']
    d, n = robe.particles.shape
    S = robe.allsettings.shape[1]
    out = dict(
        set_index=np.zeros(T, dtype=np.int64), y_meas=np.zeros((T, nch)), sigma_meas=np.zeros((T, nch)),
        resampled=np.zeros(T, dtype=np.int8), mean=np.zeros((T, d)), std=np.zeros((T, d)),
        cov=np.zeros((T, d, d)), utility=np.zeros((T, S)), n_eff=np.zeros(T),
        first_resample_step=np.int64(-1))
    worst = dict(w=0.0, util=0.0, mean=0.0, cov=0.0, part=0.0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(T):
            # ---- design half
            if sc['selection'] == 'good':
                rset = robe.good_setting()
                oset = oobe.good_setting()
                # reference does not keep the utility; recompute nothing, take the oracle's
            else:
                rset = robe.opt_setting()
                oset = oobe.opt_setting()
            assert robe.last_setting_index == oobe.last_setting_index, (sc['name'], t, 'setting index')
            assert rset == oset
            out['set_index'][t] = robe.last_setting_index
            out['utility'][t] = oobe.last_utility
            # ---- measure (simulated, shared)
            y, sig = simulate_measurement(sc, model, rset, inp, meas_rng)
            out['y_meas'][t] = y
            out['sigma_meas'][t] = sig
            ym = tuple(y) if nch > 1 else float(y[0])
            sg = tuple(sig) if nch > 1 else float(sig[0])
            record = (rset, ym, sg)
            # ---- inference half; snapshot the pre-resample weights through the oracle
            w_before = oobe.particle_weights.copy()
            p_before = oobe.particles.copy()
            robe.pdf_update(record)
            oobe.pdf_update(record)
            assert bool(robe.just_resampled) == bool(oobe.just_resampled), (sc['name'], t, 'resample flag')
            out['resampled'][t] = int(robe.just_resampled)
            if robe.just_resampled and out['first_resample_step'] < 0:
                out['first_resample_step'] = np.int64(t)
                # state right before the first resample: post-update weights of the old cloud
                if sc['kind'] == 'base':
                    lik = orc.likelihood_known_sigma(
                        (model(rset, p_before, inp['cons']),) if nch == 1 else model(rset, p_before, inp['cons']),
                        ym, sg, sc.get('choke'))
                else:
                    lik = orc.likelihood_noise_parameter(
                        (model(rset, p_before, inp['cons']),) if nch == 1 else model(rset, p_before, inp['cons']),
                        ym, p_before, sc['noise_parameter_index'], sc.get('choke'))
                out['pre_resample_weights'] = orc.normalized_product(w_before, lik)
                out['pre_resample_particles'] = p_before
                out['first_ancestors'] = oobe.last_ancestors.astype(np.int64)
                out['post_resample_particles'] = np.array(robe.particles)
            # ---- compare cloud
            rw, ow = np.asarray(robe.particle_weights), oobe.particle_weights
            # Before the first resample the restatement must match to 1e-12 relative.  After it the
            # particles agree only to ~1 ulp (the reference's numba-JITed exp and numpy's exp differ
            # by 1e-19 absolute in the weights -> covariance -> SVD factor -> last bit of the nudge),
            # and the model's conditioning (|y|/sigma * residual ~ 1e3..1e4 for c1) amplifies that
            # ulp into ~1e-12..1e-11 relative in the next weights: condition-aware 1e-9 there.
            seen_resample = out['first_resample_step'] >= 0
            # negligible weights (< 1e-15 of the largest) are compared absolutely
            np.testing.assert_allclose(ow, rw, rtol=sc.get('traj_rtol', 1e-9) if seen_resample else 1e-12,
                                       atol=1e-15 * rw.max(), err_msg=f"{sc['name']} t={t} weights")
            spread = np.std(robe.particles, axis=1, keepdims=True)
            perr = np.abs(oobe.particles - robe.particles) / (np.abs(robe.particles) * 1e-10 + spread * 1e-10)
            assert perr.max() <= 1.0, f"{sc['name']} t={t} particles differ {perr.max():.3g}x tolerance"
            worst['w'] = max(worst['w'], float(np.max(np.abs(ow - rw) / np.maximum(np.abs(rw), 1e-9 * rw.max()))))
            out['n_eff'][t] = orc.n_effective(rw)
            out['mean'][t] = robe.mean()
            out['std'][t] = robe.std()
            out['cov'][t] = robe.covariance()
            np.testing.assert_allclose(oobe.mean(), out['mean'][t], rtol=sc.get('traj_rtol', 1e-9) if seen_resample else 1e-12)
            sd = np.sqrt(np.diag(out['cov'][t]))
            cerr = np.abs(oobe.covariance() - out['cov'][t]) / np.outer(sd, sd)
            assert cerr.max() < sc.get('traj_rtol', 1e-9), f"{sc['name']} t={t} covariance {cerr.max():.3g}"
    out['final_particles'] = np.array(robe.particles)
    out['final_weights'] = np.array(robe.particle_weights)
    out['prior'] = np.array(inp['prior'])
    out['worst_weight_rel'] = np.float64(worst['w'])
    return out


def import_reference_sweeper():
    """demos/sweeper/obe_sweeper.py from the scratch copy.  The file imports matplotlib (absent here and
    irrelevant to the class): an empty stand-in module is registered first."""
    import importlib.util
    import types
    for name in ('matplotlib', 'matplotlib.pyplot'):
        sys.modules.setdefault(name, types.ModuleType(name))
    path = os.path.join(tempfile.gettempdir(), 'obe_refcopy', 'demos', 'sweeper', 'obe_sweeper.py')
    spec = importlib.util.spec_from_file_location('ref_obe_sweeper', path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.OptBayesExptSweeper


def run_sweeper_lockstep():
    """Closed loop of the sweeper demo (opt_setting -> sweep -> one pdf_update per point), reference
    against OracleSweeper, same seeds."""
    from oracle.scenarios import SWEEPER as sc
    RefSweeper = import_reference_sweeper()
    inp = build_inputs(sc)
    model = orc.MODELS[sc['model']][0]
    robe = RefSweeper(model, inp['setting_values'], inp['prior'], inp['cons'],
                      noise_parameter_index=sc['noise_parameter_index'], n_draws=sc['n_draws'], scale=sc['scale'],
                      a_param=sc['a_param'], resample_threshold=sc['resample_threshold'])
    robe.rng = np.random.default_rng(sc['seed_rng'])
    assert robe.start_stop_subsample == sc['start_stop_subsample'] and robe.cost_of_new_sweep == sc['cost_of_new_sweep']
    oobe = orc.OracleSweeper(model, inp['setting_values'], inp['prior'], inp['cons'], n_channels=1,
                             n_draws=sc['n_draws'], a_param=sc['a_param'], resample_threshold=sc['resample_threshold'],
                             scale=sc['scale'], noise_parameter_index=sc['noise_parameter_index'],
                             start_stop_subsample=sc['start_stop_subsample'],
                             cost_of_new_sweep=sc['cost_of_new_sweep'], rng=np.random.default_rng(sc['seed_rng']))
    assert np.array_equal(robe.start_stop_indices, oobe.start_stop_indices)
    meas_rng = np.random.default_rng(sc['seed_meas'])
    xvals = inp['setting_values'][0]
    T = sc['n_sweeps']
    P = len(oobe.start_stop_indices)
    d = robe.particles.shape[0]
    out = dict(pair_index=np.zeros(T, dtype=np.int64), pairs=np.zeros((T, 2), dtype=np.int64),
               sweep_utility=np.zeros((T, P)), point_utility=np.zeros((T, len(xvals))),
               mean=np.zeros((T, d)), std=np.zeros((T, d)), n_resamples=np.zeros(T, dtype=np.int64),
               start_stop_indices=np.array(oobe.start_stop_indices))
    ys = []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(T):
            state = robe.rng.bit_generator.state
            r_util = robe.sweep_utility()                 # consumes K uniforms
            robe.rng.bit_generator.state = state
            rpair = robe.opt_setting()
            opair = oobe.opt_setting()
            assert robe.last_setting_index == oobe.last_setting_index, (t, 'pair index')
            assert tuple(rpair) == tuple(opair)
            seen = t > 0
            np.testing.assert_allclose(oobe.last_sweep_utility, r_util, rtol=sc['traj_rtol'] if seen else 1e-12)
            out['pair_index'][t] = oobe.last_setting_index
            out['pairs'][t] = opair
            out['sweep_utility'][t] = oobe.last_sweep_utility
            out['point_utility'][t] = oobe.last_utility
            start, stop = int(rpair[0]), int(rpair[1])
            sweep_x = xvals[start:stop]
            y_true = model((sweep_x,), sc['true_pars'], inp['cons'])
            y = y_true + sc['noise'] * meas_rng.standard_normal(len(sweep_x))
            ys.append(y)
            n_res = 0
            # the reference's pdf_update loops over the points; count its resamples point by point
            for xs, yv in zip(sweep_x, y):
                robe.pdf_update(((np.array([xs]),), np.array([yv])))
                oobe.pdf_update(((np.array([xs]),), np.array([yv])))
                assert bool(robe.just_resampled) == bool(oobe.just_resampled), (t, 'resample flag')
                n_res += int(robe.just_resampled)
            out['n_resamples'][t] = n_res
            out['mean'][t] = robe.mean()
            out['std'][t] = robe.std()
            np.testing.assert_allclose(oobe.mean(), out['mean'][t], rtol=sc['traj_rtol'])
            np.testing.assert_allclose(oobe.particle_weights, robe.particle_weights, rtol=sc['traj_rtol'],
                                       atol=1e-15 * robe.particle_weights.max())
    out['y_concat'] = np.concatenate(ys)
    out['y_lengths'] = np.array([len(v) for v in ys], dtype=np.int64)
    out['prior'] = np.array(inp['prior'])
    out['final_particles'] = np.array(robe.particles)
    out['final_weights'] = np.array(robe.particle_weights)
    return out


#: keys of a run_lockstep() record that are recorded for diagnosis only: neither tests/test_oracle.py nor
#: tests/test_gpu_parity.py reads them.  (The sweeper record is stored whole: tests/test_gpu_sweeper.py reads its std.)
DIAGNOSTIC_KEYS = ('std', 'n_eff', 'first_resample_step', 'pre_resample_weights', 'pre_resample_particles',
                   'post_resample_particles', 'worst_weight_rel')
#: a utility row longer than this is stored at a fixed, seeded sample of the settings (utility_columns)
MAX_UTILITY_COLUMNS = 4096


def shrink(out):
    """A scenario's golden record as stored: the diagnostic keys dropped, and a long utility row (c3's 101 x 101 grid)
    sampled at MAX_UTILITY_COLUMNS fixed settings that include every chosen one.  The chosen indices themselves
    are still checked against the whole grid (set_index)."""
    keep = {k: v for k, v in out.items() if k not in DIAGNOSTIC_KEYS}
    util = keep.get('utility')
    if util is not None and util.shape[1] > MAX_UTILITY_COLUMNS:
        cols = np.random.default_rng(0).choice(util.shape[1], MAX_UTILITY_COLUMNS, replace=False)
        cols = np.unique(np.concatenate((cols, keep['set_index']))).astype(np.int64)
        keep['utility'] = util[:, cols]
        keep['utility_columns'] = cols
    return keep


def check_equivalences():
    """The numpy identities the oracle relies on (SURVEY 8c), re-verified against this numpy."""
    rng = np.random.default_rng(7)
    w = rng.random(5000)
    w /= w.sum()
    for m in (1, 30, 5000):
        g1 = np.random.default_rng(11)
        g2 = np.random.default_rng(11)
        a = g1.choice(np.arange(5000), size=m, p=w)
        b = orc.choice_indices(w, g2.random(m))
        assert np.array_equal(a, b), 'choice equivalence'
        assert g1.random() == g2.random(), 'generator state after choice'
    cov = np.cov(rng.standard_normal((3, 200)))
    g1 = np.random.default_rng(5)
    g2 = np.random.default_rng(5)
    a = g1.multivariate_normal(np.zeros(3), cov, 1000)
    b = g2.standard_normal(3000).reshape(1000, 3) @ orc.mvn_factor_svd(cov)
    assert np.array_equal(a, b), 'multivariate_normal svd restatement must be bit-equal'
    x = rng.standard_normal((3, 400))
    ww = rng.random(400)
    np.testing.assert_allclose(orc.weighted_covariance_formula(x, ww), np.cov(x, aweights=ww), rtol=1e-12)
    assert np.array_equal(orc.weighted_mean(x, ww), np.average(x, axis=1, weights=ww))
    print('numpy equivalences: OK')


def check_entropy_utilities(ref):
    """utility_pseudo / utility_full_kld of the reference against the oracle on the same draws."""
    from oracle.scenarios import by_name
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc, 4000)
    model = orc.MODELS[sc['model']][0]
    for method in ('pseudo_utility', 'full_kld_utility'):
        obe = ref.OptBayesExpt(model, inp['setting_values'], inp['prior'], inp['cons'], utility_method=method,
                               default_noise_std=500.0, n_draws=30)
        obe.rng = np.random.default_rng(17)
        ref.obe_base.rng = np.random.default_rng(23)
        got = np.asarray(obe.utility())
        g = np.random.default_rng(17)
        draws, _ = orc.randdraw(inp['prior'], np.ones(4000) / 4000, g.random(30))
        _, ys = orc.yvar_from_draws(model, orc.make_allsettings(inp['setting_values']), draws, inp['cons'], 1)
        if method == 'pseudo_utility':
            want = orc.utility_pseudo(ys, orc.noise_var_default(500.0, 1))
        else:
            nva = np.random.default_rng(23).normal(0, 1.0, 30).reshape((1, 30))
            noise = (nva * np.sqrt(orc.noise_var_default(500.0, 1))).T
            want = orc.utility_full_kld(ys, noise)
        np.testing.assert_allclose(got, want, rtol=1e-13, err_msg=method)
        for n_draws in (8, 30):   # van Es (n <= 10) and Ebrahimi branches of the estimator
            pass
    print('entropy utilities: OK')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reference', required=True, help='source tree of usnistgov/optbayesexpt v1.2.0')
    ap.add_argument('--check', action='store_true')
    ap.add_argument('--only', default=None)
    args = ap.parse_args()
    ref = import_reference(args.reference)
    check_equivalences()
    check_entropy_utilities(ref)
    os.makedirs(GOLDEN, exist_ok=True)
    for sc in SCENARIOS:
        if args.only and sc['name'] != args.only:
            continue
        out = run_lockstep(ref, sc)
        print(f"{sc['name']}: lock-step OK over {sc['n_cycles']} cycles, "
              f"{int(out['resampled'].sum())} resamples, worst weight rel diff {out['worst_weight_rel']:.2e}")
        if not args.check:
            keep = shrink(out)
            if not sc.get('store_prior', True):
                keep.pop('prior')
                keep.pop('pre_resample_particles', None)
            np.savez_compressed(os.path.join(GOLDEN, f"{sc['name']}.npz"), **keep)
    if not args.only or args.only == 'sweeper_lorentzian':
        out = run_sweeper_lockstep()
        print(f"sweeper_lorentzian: lock-step OK over {len(out['pair_index'])} sweeps "
              f"({int(out['y_lengths'].sum())} point updates, {int(out['n_resamples'].sum())} resamples)")
        if not args.check:
            np.savez_compressed(os.path.join(GOLDEN, 'sweeper_lorentzian.npz'), **out)
    print('all scenarios pinned')


if __name__ == '__main__':
    main()
