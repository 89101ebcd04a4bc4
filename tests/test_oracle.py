"""CPU tests of the oracle: (1) every known-answer assertion the reference's own tests hold for
this path, replayed against oracle/obe_oracle.py; (2) the committed golden trajectories (written
by oracle/pin_against_reference.py from the UNMODIFIED reference) replayed by the oracle with no
reference present."""
import os

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import obe_oracle as orc
from oracle.scenarios import SCENARIOS, build_inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PRIOR4 = np.array([[0., 1., 2., 3.], [1., 3., 2., 4.]])


# ---- reference tests/test_particlepdf.py ---------------------------------------------------
def test_mean_known_answer():                       # tests/test_particlepdf.py:69-77
    w = np.ones(4) / 4
    assert_array_equal(orc.weighted_mean(PRIOR4, w), np.array([1.5, 2.5]))


def test_covariance_known_answer():                 # tests/test_particlepdf.py:80-90
    w = np.ones(4) / 4
    expect = np.array([[5, 4], [4, 5]]) / 3
    assert_allclose(orc.weighted_covariance(PRIOR4, w), expect)
    assert_allclose(orc.weighted_covariance_formula(PRIOR4, w), expect)


def test_std_known_answer():                        # tests/test_particlepdf.py:93-102
    w = np.ones(4) / 4
    assert_array_equal(orc.std_biased(PRIOR4, w), np.sqrt(np.array([5, 5]) / 4))


def test_bayesian_update_known_answer():            # tests/test_particlepdf.py:105-117
    lik = np.array([1., 2., 3., 4.])
    w = orc.normalized_product(np.ones(4) / 4, lik)
    assert_array_equal(w, lik / np.sum(lik))


def test_resample_test_thresholds():                # tests/test_particlepdf.py:138-152
    assert orc.resample_decision(np.array([.1, .4, .4, .1]), 0.5)[0] is False
    assert orc.resample_decision(np.array([0, .75, .25, 0]), 0.5)[0] is True


def test_resample_shapes_and_uniform_weights():     # tests/test_particlepdf.py:125-135
    rng = np.random.default_rng(0)
    new, w, idx = orc.resample(PRIOR4, np.array([.1, .4, .4, .1]), rng.random(4), rng.standard_normal(8))
    assert new.shape == (2, 4) and idx.shape == (4,)
    assert_array_equal(w, np.ones(4) / 4)


# ---- reference tests/test_optbayesexpt.py --------------------------------------------------
def _fakefunc(sets, pars, cons):
    x, = sets
    a, b = pars
    return a + b * x


def test_allsettings_and_model_orientations():      # tests/test_optbayesexpt.py:21-44
    alls = orc.make_allsettings((np.array([0, 1, 2]),))
    assert_array_equal(alls, [[0, 1, 2]])
    assert_array_equal(_fakefunc((1,), PRIOR4, ()), [1, 4, 4, 7])
    assert_array_equal(_fakefunc(alls, [1, 3], ()), [1, 4, 7])   # the reference wraps it into a 1-tuple


def test_likelihood_known_answer():                 # tests/test_optbayesexpt.py:47-55
    ymodel = np.array(((1., 4., 4., 7.),))
    lkl = np.exp(-(ymodel - 5.0) ** 2 / 2)[0]
    assert_array_equal(orc.likelihood_known_sigma(ymodel, (5.0,), 1.0), lkl)


def test_pdf_update_known_answer():                 # tests/test_optbayesexpt.py:58-69
    eng = orc.OracleOBE(_fakefunc, (np.array([0, 1, 2]),), PRIOR4, ())
    eng.pdf_update(((1,), 5.0, 1.0))
    lkl = np.exp(-(np.array((1., 4., 4., 7.)) - 5.0) ** 2 / 2)
    assert_array_equal(eng.particle_weights, lkl / np.sum(lkl))


# ---- reference tests/test_zinference.py::test_infer -----------------------------------------
def test_infer_analytic_posterior():                # tests/test_zinference.py:89-108
    n, true_mean, true_sigma = 5000, 2.0, 1.5
    x = np.linspace(-5, 5, n)
    eng = orc.OracleOBE(lambda s, p, c: p[0], (), np.array([x, np.ones(n) * true_sigma]), (),
                        resample_threshold=0.0)
    eng.allsettings = np.zeros((0, 1))
    eng.pdf_update(((), true_mean, true_sigma))
    post = np.exp(-(true_mean - x) ** 2 / (2 * true_sigma ** 2)) / (np.sqrt(2 * np.pi) * true_sigma)
    post /= post.sum()
    assert_allclose(eng.particle_weights, post, atol=1e-15, rtol=1e-15)


# ---- properties of the restated pieces --------------------------------------------------------
def test_choice_equals_generator_choice():
    rng = np.random.default_rng(3)
    w = rng.random(1000)
    w /= w.sum()
    g1, g2 = np.random.default_rng(9), np.random.default_rng(9)
    assert_array_equal(g1.choice(np.arange(1000), size=1000, p=w), orc.choice_indices(w, g2.random(1000)))


def test_systematic_comb_is_monotone_and_in_range():
    for n in (1, 7, 2048, 100003):
        for u0 in (0.0, 0.5, np.nextafter(1.0, 0.0)):
            u = orc.systematic_uniforms(u0, n)
            assert np.all(np.diff(u) >= 0) and u[0] >= 0
            w = np.random.default_rng(n).random(n)
            idx = orc.search_cdf(orc.normalized_cdf(w), u)
            assert idx.min() >= 0 and idx.max() <= n - 1 and np.all(np.diff(idx) >= 0)


def test_philox_known_answer():
    # Random123 known-answer vectors for philox4x32-10
    out = orc.philox4x32_10(np.uint32(0), np.uint32(0), np.uint32(0), np.uint32(0), 0, 0)
    assert [int(x) for x in out] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    out = orc.philox4x32_10(np.uint32(0xffffffff), np.uint32(0xffffffff), np.uint32(0xffffffff),
                            np.uint32(0xffffffff), 0xffffffff, 0xffffffff)
    assert [int(x) for x in out] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    out = orc.philox4x32_10(np.uint32(0x243f6a88), np.uint32(0x85a308d3), np.uint32(0x13198a2e),
                            np.uint32(0x03707344), 0xa4093822, 0x299f31d0)
    assert [int(x) for x in out] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_device_normals_are_standard_normal():
    z = orc.device_normals(200000, 3, 12345, 1)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    assert abs(np.corrcoef(z.T)[0, 1]) < 0.01


def test_packed_device_normals():
    """The packed stream of the streaming resample kernels: standard normal, independent of how the slots are cut
    into ranges (sharding invariance), and every Philox word used exactly once."""
    z = orc.device_normals_packed(200000, 3, 12345, 1)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    assert abs(np.corrcoef(z.T)[0, 1]) < 0.01 and abs(np.corrcoef(z[:-1, 2], z[1:, 0])[0, 1]) < 0.01
    for d in (1, 2, 3, 5, 8):
        whole = orc.device_normals_packed(1000, d, 99, 4)
        assert_array_equal(whole[337:911], orc.device_normals_packed(911 - 337, d, 99, 4, slot_begin=337))
        assert len(np.unique(whole)) >= whole.size - 4          # (23-bit uniforms: a chance collision is possible)
    assert not np.array_equal(orc.device_normals_packed(64, 3, 99, 4), orc.device_normals_packed(64, 3, 99, 5))


def test_mvn_factors_reproduce_covariance():
    cov = np.array([[2.0, 0.3, 0.1], [0.3, 1.0, -0.2], [0.1, -0.2, 0.5]])
    for f in (orc.mvn_factor_svd(cov), orc.mvn_factor_cholesky(cov)):
        assert_allclose(f.T @ f, cov, atol=1e-14)


# ---- golden trajectories of the unmodified reference, replayed by the oracle ------------------
@pytest.mark.parametrize('sc', SCENARIOS, ids=[s['name'] for s in SCENARIOS])
def test_oracle_replays_reference_golden(sc):
    g = np.load(os.path.join(GOLDEN, sc['name'] + '.npz'))
    inp = build_inputs(sc)
    assert_array_equal(inp['prior'], g['prior'])        # seeded inputs regenerate bit-identically
    model, _, _, _, nch = orc.MODELS[sc['model']]
    eng = orc.OracleOBE(model, inp['setting_values'], inp['prior'], inp['cons'], n_channels=nch,
                        n_draws=sc['n_draws'], choke=sc.get('choke'), pickiness=sc.get('pickiness', 15),
                        default_noise_std=sc.get('default_noise_std', 1.0), a_param=sc['a_param'],
                        resample_threshold=sc['resample_threshold'], scale=sc['scale'],
                        noise_parameter_index=sc.get('noise_parameter_index'),
                        nonneg_constraint=(sc['kind'] == 'lockin'),
                        cost_of_changing_setting=sc.get('cost_of_changing_setting'),
                        rng=np.random.default_rng(sc['seed_rng']))
    tol = sc.get('traj_rtol', 1e-9)
    cols = g['utility_columns'] if 'utility_columns' in g.files else slice(None)   # (a large grid is sampled)
    seen = False
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(sc['n_cycles']):
            setting = eng.good_setting() if sc['selection'] == 'good' else eng.opt_setting()
            assert eng.last_setting_index == g['set_index'][t], f't={t}'
            assert_allclose(eng.last_utility[cols], g['utility'][t], rtol=tol if seen else 1e-12)
            y, sig = g['y_meas'][t], g['sigma_meas'][t]
            rec = (setting, tuple(y) if nch > 1 else float(y[0]), tuple(sig) if nch > 1 else float(sig[0]))
            eng.pdf_update(rec)
            assert int(eng.just_resampled) == g['resampled'][t], f't={t}'
            if eng.just_resampled and not seen:
                assert_array_equal(eng.last_ancestors, g['first_ancestors'])
            seen = seen or eng.just_resampled
            assert_allclose(eng.mean(), g['mean'][t], rtol=tol if seen else 1e-12)
    assert_allclose(eng.particle_weights, g['final_weights'], rtol=max(tol, 1e-9),
                    atol=1e-15 * g['final_weights'].max())


def test_golden_shrink_keeps_what_the_replays_read():
    """oracle/pin_against_reference.py stores every scenario record through shrink(): it must keep each key that the
    replays here and in tests/test_gpu_parity.py read."""
    from oracle.pin_against_reference import shrink
    read = {'prior', 'set_index', 'utility', 'y_meas', 'sigma_meas', 'resampled', 'first_ancestors', 'mean', 'cov',
            'final_weights', 'final_particles'}
    for sc in SCENARIOS:
        g = np.load(os.path.join(GOLDEN, sc['name'] + '.npz'))
        assert read <= set(g.files) and read <= set(shrink({k: g[k] for k in g.files})), sc['name']


# ---- sweeper workload (demos/sweeper/obe_sweeper.py), SURVEY 8(f) row 2 ------------------------------
def test_sweep_pairs_and_utility_known_answer():
    pairs = orc.sweep_start_stop_indices(8, 3)              # subsamples 0, 3, 6 + the last index 7
    assert_array_equal(pairs, [[0, 3], [0, 6], [0, 7], [3, 6], [3, 7], [6, 7]])
    u = np.arange(1.0, 9.0)                                 # cumsum = 1, 3, 6, 10, 15, 21, 28, 36
    su = orc.sweep_utility(u, pairs, 5.0)
    assert_allclose(su, [(10 - 1) / 8, (28 - 1) / 11, (36 - 1) / 12, (28 - 10) / 8, (36 - 10) / 9, (36 - 28) / 6],
                    rtol=1e-15)


def test_oracle_sweeper_replays_reference_golden():
    from oracle.scenarios import SWEEPER as sc
    g = np.load(os.path.join(GOLDEN, sc['name'] + '.npz'))
    inp = build_inputs(sc)
    assert_array_equal(inp['prior'], g['prior'])
    model = orc.MODELS[sc['model']][0]
    eng = orc.OracleSweeper(model, inp['setting_values'], inp['prior'], inp['cons'], n_channels=1,
                            n_draws=sc['n_draws'], a_param=sc['a_param'], resample_threshold=sc['resample_threshold'],
                            scale=sc['scale'], noise_parameter_index=sc['noise_parameter_index'],
                            start_stop_subsample=sc['start_stop_subsample'], cost_of_new_sweep=sc['cost_of_new_sweep'],
                            rng=np.random.default_rng(sc['seed_rng']))
    assert_array_equal(eng.start_stop_indices, g['start_stop_indices'])
    xvals = inp['setting_values'][0]
    ofs = np.concatenate(([0], np.cumsum(g['y_lengths'])))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(sc['n_sweeps']):
            pair = eng.opt_setting()
            assert eng.last_setting_index == g['pair_index'][t], f't={t}'
            assert_array_equal(pair, g['pairs'][t])
            assert_allclose(eng.last_sweep_utility, g['sweep_utility'][t], rtol=sc['traj_rtol'] if t else 1e-12)
            y = g['y_concat'][ofs[t]:ofs[t + 1]]
            eng.pdf_update(((xvals[pair[0]:pair[1]],), y))
            assert_allclose(eng.mean(), g['mean'][t], rtol=sc['traj_rtol'])
    assert_allclose(eng.particle_weights, g['final_weights'], rtol=sc['traj_rtol'],
                    atol=1e-15 * g['final_weights'].max())
