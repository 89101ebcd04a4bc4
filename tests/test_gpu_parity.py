"""GPU parity tests: the CUDA path, called through the C ABI / the mirrored classes, against the
numpy oracle on identical seeded inputs, against the reference's own known answers, and against
the golden trajectories recorded from the unmodified reference.

Tolerances (north_star): likelihood / weights / moments / utility 1e-12 relative in fp64
(condition-aware where the reference's own value is ill-conditioned); ancestor indices bit-exact
given the same uniforms; chosen setting index identical.
"""
import ctypes as C
import os
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import obe_oracle as orc
from oracle.scenarios import SCENARIOS, build_inputs, by_name

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PRIOR4 = (np.array([0., 1., 2., 3.]), np.array([1., 3., 2., 4.]))


@pytest.fixture(scope='module')
def obe():
    import optbayesexpt_b200 as pkg
    return pkg


@pytest.fixture(scope='module')
def torch():
    import torch as t
    assert t.cuda.is_available(), 'GPU tests need a CUDA device'
    return t


def wclose(actual, desired, rtol=1e-12, msg=''):
    """weights: relative, with an absolute floor for weights < 1e-15 of the largest"""
    assert_allclose(actual, desired, rtol=rtol, atol=1e-15 * np.max(np.abs(desired)), err_msg=msg)


def cov_close(actual, desired, tol):
    sd = np.sqrt(np.diag(desired))
    err = np.abs(actual - desired) / np.outer(sd, sd)
    assert err.max() < tol, f'covariance off by {err.max():.3g} (correlation units)'


# =================================================================================================
# 1. the reference's own tests, run against the mirrored classes
# =================================================================================================
def test_ref_particlepdf_init_and_set_pdf(obe):                 # tests/test_particlepdf.py:17-61
    pdf = obe.ParticlePDF(PRIOR4)
    assert pdf.n_dims == 2 and pdf.n_particles == 4
    assert_array_equal(np.asarray([[0, 1, 2, 3], [1, 3, 2, 4]]), pdf.particles)
    assert_array_equal([.25, .25, .25, .25], pdf.particle_weights)
    assert pdf.just_resampled is False
    samples = np.arange(15).reshape((3, 5))
    pdf.set_pdf(samples)
    assert pdf.n_dims == 3 and pdf.n_particles == 5
    assert_array_equal(samples, pdf.particles)
    assert_array_equal(np.ones(5) / 5.0, pdf.particle_weights)
    ww = np.array([1, 2, 3, 4, 5])
    pdf.set_pdf(samples, weights=ww)
    assert_array_equal(ww / np.sum(ww), pdf.particle_weights)
    with pytest.raises(ValueError):
        pdf.set_pdf(samples, weights=np.array([1, 2, 3]))


def test_ref_particlepdf_moments(obe):                          # tests/test_particlepdf.py:69-102
    pdf = obe.ParticlePDF(PRIOR4)
    assert_allclose(pdf.mean(), np.array([1.5, 2.5]), rtol=1e-15)
    assert_allclose(pdf.covariance(), np.array([[5, 4], [4, 5]]) / 3, rtol=1e-14)
    assert_allclose(pdf.std(), np.sqrt(np.array([5, 5]) / 4), rtol=1e-15)
    one = obe.ParticlePDF((np.array([0., 1., 2., 3.]),))
    assert one.covariance().shape == (1, 1)                      # particlepdf.py:195-196


def test_ref_particlepdf_bayesian_update(obe):                  # tests/test_particlepdf.py:105-117
    pdf = obe.ParticlePDF(PRIOR4)
    pdf.tuning_parameters['auto_resample'] = False
    lik = np.array([1., 2., 3., 4.])
    pdf.bayesian_update(lik)
    assert_allclose(pdf.particle_weights, lik / np.sum(lik), rtol=1e-15)


@pytest.mark.parametrize('mode', ['systematic', 'multinomial'])
def test_ref_particlepdf_resample(obe, mode):                   # tests/test_particlepdf.py:125-152
    pdf = obe.ParticlePDF(PRIOR4, resampling=mode, seed=5)
    pdf.particle_weights = np.array([.1, .4, .4, .1])
    pdf.resample()
    assert pdf.particles.shape == (2, 4)
    assert_array_equal(pdf.particle_weights, np.ones(4) / 4)
    pdf = obe.ParticlePDF(PRIOR4, resampling=mode, seed=5)
    pdf.particle_weights = np.array([.1, .4, .4, .1])
    pdf.resample_test()
    assert pdf.just_resampled is False
    pdf.particle_weights = np.array([0, .75, .25, 0])
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        pdf.resample_test()
    assert pdf.just_resampled is True


LINE_AB = '''
__device__ void fake_model(const double* s, const double* p, const double* c, double* y) {
    y[0] = obe_add(p[0], obe_mul(p[1], s[0]));   // a + b*x   (tests/test_optbayesexpt.py:10-13)
}
'''


def _fake_obe(obe):
    model = obe.cuda_source(LINE_AB, 'fake_model', n_settings=1, n_params=2)
    return obe.OptBayesExpt(model, (np.array([0, 1, 2]),), PRIOR4, ())


def test_ref_optbayesexpt_init_and_model(obe):                  # tests/test_optbayesexpt.py:21-44 (NVRTC model)
    eng = _fake_obe(obe)
    assert_array_equal((np.array([0, 1, 2]),), eng.allsettings)
    assert_array_equal(PRIOR4, eng.parameters)
    assert_array_equal([[1, 4, 4, 7]], eng.eval_over_all_parameters((1,)))
    assert_array_equal([[1, 4, 7]], eng.eval_over_all_settings([1, 3]))


def test_ref_optbayesexpt_likelihood_and_update(obe):           # tests/test_optbayesexpt.py:47-69
    eng = _fake_obe(obe)
    ymodel = np.array(((1., 4., 4., 7.),))
    lkl = np.exp(-(ymodel - 5.0) ** 2 / 2)[0]
    assert_allclose(eng.likelihood(ymodel, ((1,), (5.0,), 1.0)), lkl, rtol=2e-16)
    eng.pdf_update(((1,), 5.0, 1.0))
    assert_allclose(eng.particle_weights, lkl / np.sum(lkl), rtol=1e-15)
    # precomputed model data path (obe_base.py:374-385)
    eng2 = _fake_obe(obe)
    eng2.pdf_update(((1,), 5.0, 1.0), y_model_data=ymodel)
    assert_allclose(eng2.particle_weights, lkl / np.sum(lkl), rtol=1e-15)
    # ... and with the model pass prefetched on the device (no host round trip)
    eng3 = _fake_obe(obe)
    ydev = eng3.eval_over_all_parameters_dev((1,))
    assert ydev.is_cuda and ydev.shape[0] == 1
    eng3.pdf_update(((1,), 5.0, 1.0), y_model_data=ydev)
    assert_allclose(eng3.particle_weights, lkl / np.sum(lkl), rtol=1e-15)


def test_prefetched_model_pass_equals_fused_update(obe):
    """prefetch_model(setting) -> pdf_update(record) uses the model values computed ahead (side stream) and gives
    the same posterior as the fused pass; a resample in between invalidates the prefetch."""
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc, 50000)
    kw = dict(scale=False, default_noise_std=500.0, seed=5)
    a = obe.OptBayesExpt(sc['model'], inp['setting_values'], inp['prior'], inp['cons'], **kw)
    b = obe.OptBayesExpt(sc['model'], inp['setting_values'], inp['prior'], inp['cons'], **kw)
    rec = ((3.05,), 49500.0, 500.0)
    a.prefetch_model(rec[0])
    assert a._prefetched is not None
    a.pdf_update(rec)
    assert a._prefetched is None
    b.pdf_update(rec)
    # the prefetch evaluates the exact functor, the fused pass the update-pass variant: last-bit differences
    wclose(a.particle_weights, b.particle_weights, 1e-12)
    assert_allclose(a.mean(), b.mean(), rtol=1e-12)
    # stale prefetch: wrong setting, or the cloud changed
    a.prefetch_model((2.0,))
    a.pdf_update(rec)
    b.pdf_update(rec)
    wclose(a.particle_weights, b.particle_weights, 1e-12)
    a.prefetch_model(rec[0])
    a.resample()
    b.resample()
    assert a._take_prefetched(rec[0]) is None


def test_ref_zinference_infer(obe):                             # tests/test_zinference.py:89-108
    n, true_mean, true_sigma = 5000, 1.0, 1.0
    src = '__device__ void ident(const double* s, const double* p, const double* c, double* y) { y[0] = p[0]; }'
    model = obe.cuda_source(src, 'ident', n_settings=1, n_params=1, n_constants=1)
    x = np.linspace(-5, 5, n)
    eng = obe.OptBayesExpt(model, (0,), (x, np.ones(n) * true_sigma), (0,))
    eng.tuning_parameters['resample_threshold'] = 0
    eng.pdf_update(((), true_mean, true_sigma))
    post = np.exp(-(true_mean - x) ** 2 / (2 * true_sigma ** 2)) / (np.sqrt(2 * np.pi) * true_sigma)
    post /= np.sum(post)
    assert_allclose(eng.particle_weights, post, atol=1e-15, rtol=1e-15)


def test_error_behaviour(obe):
    with pytest.raises(SyntaxError):                             # obe_base.py:242
        obe.OptBayesExpt('line', (np.linspace(0, 1, 5),), PRIOR4, (), utility_method='nope')
    with pytest.raises(SyntaxError):                             # obe_base.py:254
        obe.OptBayesExpt('line', (np.linspace(0, 1, 5),), PRIOR4, (), selection_method='nope')
    with pytest.raises(RuntimeError):                            # obe_noiseparam.py:53-55
        obe.OptBayesExptNoiseParameter('lockin_coil', (np.linspace(1, 2, 5),),
                                       np.ones((4, 8)), (), noise_parameter_index=3)
    with pytest.raises(TypeError):
        obe.OptBayesExpt(lambda s, p, c: 0, (np.linspace(0, 1, 5),), PRIOR4, ())
    pdf = obe.ParticlePDF(PRIOR4)
    with pytest.raises(ValueError):
        pdf.particles[0, 0] = 7.0                                # mirrors are read-only: loud, not silent


# =================================================================================================
# 2. kernel-level parity against the oracle
# =================================================================================================
def _engine(obe, sc, n=None, **kw):
    inp = build_inputs(sc, n)
    args = dict(n_draws=sc['n_draws'], scale=sc['scale'], a_param=sc['a_param'],
                resample_threshold=sc['resample_threshold'], resampling='multinomial')
    if sc.get('choke') is not None:
        args['choke'] = sc['choke']
    args.update(kw)
    if sc['kind'] == 'base':
        eng = obe.OptBayesExpt(sc['model'], inp['setting_values'], inp['prior'], inp['cons'],
                               default_noise_std=sc.get('default_noise_std', 1.0), **args)
    elif sc['kind'] == 'noise':
        eng = obe.OptBayesExptNoiseParameter(sc['model'], inp['setting_values'], inp['prior'], inp['cons'],
                                             noise_parameter_index=sc['noise_parameter_index'], **args)
    else:
        class Lockin(obe.OptBayesExptNoiseParameter):           # demos/lockin/lockin_of_coil.py:107-153
            cost_of_changing_setting = sc['cost_of_changing_setting']

            def enforce_parameter_constraints(self):
                self._apply_constraint_masks(mask_lt=(1 << self.n_dims) - 1)

            def cost_estimate(self):
                cost = np.ones_like(self.allsettings[0]) * self.cost_of_changing_setting
                cost[self.last_setting_index] = 1.0
                return cost
        eng = Lockin(sc['model'], inp['setting_values'], inp['prior'], inp['cons'],
                     noise_parameter_index=sc['noise_parameter_index'], **args)
    eng.rng = np.random.default_rng(sc['seed_rng'])
    return eng, inp


def _oracle_update(sc, inp, particles, w, record):
    model, _, _, _, nch = orc.MODELS[sc['model']]
    y = model(record[0], particles, inp['cons'])
    y = y if nch > 1 else (y,)
    if sc['kind'] == 'base':
        lik = orc.likelihood_known_sigma(y, record[1], record[2], sc.get('choke'))
    else:
        lik = orc.likelihood_noise_parameter(y, record[1], particles, sc['noise_parameter_index'], sc.get('choke'))
    return orc.normalized_product(w, lik), lik


RECORDS = {
    'c1_find_peak': ((3.0,), 49500.0, 500.0),
    'c1_good_scale': ((2.9,), 49300.0, 500.0),
    'c2_line_noise': ((0.4,), 0.1),
    'c3_pipulse': ((0.31, 1.2), 99700.0, 315.0),
    'c5_lockin': ((2 * np.pi * 3000.0,), (9.0, 21.0)),
}


@pytest.mark.parametrize('name', list(RECORDS))
@pytest.mark.parametrize('n', [10000, 12345, 1])
def test_update_matches_oracle(obe, name, n):
    sc = by_name(name)
    eng, inp = _engine(obe, sc, n)
    eng.tuning_parameters['auto_resample'] = False
    rec = RECORDS[name]
    if sc['kind'] != 'base':
        rec = (rec[0], rec[1], None)
    w0 = np.ones(n) / n
    w1, lik = _oracle_update(sc, inp, inp['prior'], w0, rec)
    eng.pdf_update(rec)
    wclose(eng.particle_weights, w1, 1e-12, 'first update')
    # a second update on top of non-uniform weights (exercises the lazy normaliser)
    rec2 = (rec[0], tuple(np.atleast_1d(rec[1]) * 1.001) if np.ndim(rec[1]) else rec[1] * 1.001, rec[2])
    w2, _ = _oracle_update(sc, inp, inp['prior'], w1, rec2)
    eng.pdf_update(rec2)
    wclose(eng.particle_weights, w2, 1e-12, 'second update')
    if np.sum(w2) > 0:                                           # a lone particle can underflow to 0/0
        assert_allclose(eng.n_eff(), orc.n_effective(w2), rtol=1e-12)
    if n > 1:
        assert_allclose(eng.mean(), orc.weighted_mean(inp['prior'], w2), rtol=1e-12)
        cov_close(eng.covariance(), orc.weighted_covariance_longdouble(inp['prior'], w2), 1e-12)
        assert_allclose(eng.std(), orc.std_biased_longdouble(inp['prior'], w2), rtol=1e-11)
    if sc['kind'] != 'base' and np.sum(w2) > 0:
        assert_allclose(eng.yvar_noise_model(),
                        orc.noise_var_noise_parameter(inp['prior'], w2, sc['noise_parameter_index']), rtol=1e-12)


def test_update_large_matches_oracle(obe):
    """N = 1e6 (config c3 size), Lorentzian: the oracle still finishes in well under a second."""
    sc = by_name('c1_find_peak')
    n = 1000000
    eng, inp = _engine(obe, sc, n)
    eng.tuning_parameters['auto_resample'] = False
    rec = RECORDS['c1_find_peak']
    w1, _ = _oracle_update(sc, inp, inp['prior'], np.ones(n) / n, rec)
    eng.pdf_update(rec)
    wclose(eng.particle_weights, w1, 1e-12)
    assert_allclose(eng.mean(), orc.weighted_mean(inp['prior'], w1), rtol=1e-12)
    cov_close(eng.covariance(), orc.weighted_covariance_longdouble(inp['prior'], w1), 1e-12)


def test_nan_to_num_semantics(obe):
    """zero / tiny sigma drives the likelihood to inf/nan: weights must follow numpy.nan_to_num
    (particlepdf.py:137-138)."""
    eng = obe.OptBayesExpt('line', (np.linspace(0, 1, 5),), (np.array([0., 1., 2., 3.]), np.array([1., 3., 2., 4.])),
                           (), resampling='multinomial')
    eng.tuning_parameters['auto_resample'] = False
    rec = ((1.0,), 4.0, 1e-200)
    y = orc.model_line(rec[0], np.array(PRIOR4), ())
    with np.errstate(all='ignore'):
        lik = orc.likelihood_known_sigma((y,), rec[1], rec[2])
        want = orc.normalized_product(np.ones(4) / 4, lik)
    eng.pdf_update(rec)
    assert_allclose(eng.particle_weights, want, rtol=1e-12, atol=0)


@pytest.mark.parametrize('n', [5000, 2048, 2049, 1000000])
def test_cdf_search_and_draws(obe, torch, n):
    """(a) idx == searchsorted(cdf_gpu, u, 'right') bit-exact; (b) cdf_gpu == cumsum to 1e-12;
    (c) vs the reference's own indices: mismatches counted, must be 0 here."""
    from optbayesexpt_b200 import _lib
    rng = np.random.default_rng(n)
    pdf = obe.ParticlePDF(rng.standard_normal((3, n)), resampling='multinomial')
    w = rng.random(n) ** 3
    w /= w.sum()
    pdf.particle_weights = w
    lib = _lib.load()
    cdf = torch.empty(n, dtype=torch.float64, device='cuda')
    _lib.check(lib.obe_cdf(pdf._cs(), C.c_void_p(cdf.data_ptr()), pdf._stream()))
    cdf_h = cdf.cpu().numpy()
    assert cdf_h[-1] == 1.0
    assert np.all(np.diff(cdf_h) >= 0)
    assert_allclose(cdf_h, orc.normalized_cdf(w), rtol=1e-12)
    m = min(n, 200000)
    u = rng.random(m)
    u_dev = torch.from_numpy(u).cuda()
    idx = torch.empty(m, dtype=torch.int64, device='cuda')
    _lib.check(lib.obe_search(pdf._cs(), C.c_void_p(cdf.data_ptr()), C.c_void_p(u_dev.data_ptr()), m,
                              C.c_void_p(idx.data_ptr()), pdf._stream()))
    idx_h = idx.cpu().numpy()
    assert_array_equal(idx_h, orc.search_cdf(cdf_h, u))                      # (a)
    mism = int(np.sum(idx_h != orc.choice_indices(w, u)))                      # (c)
    assert mism == 0, f'{mism} ancestors differ from the reference cumsum path'
    # K draws without a materialised CDF
    k = 30
    pdf.rng = np.random.default_rng(77)
    uk = np.random.default_rng(77).random(k)
    draws = pdf.randdraw(k)
    want_idx = orc.search_cdf(cdf_h, uk)
    assert_array_equal(draws, pdf.particles[:, want_idx])
    assert_array_equal(want_idx, orc.choice_indices(w, uk))


def test_draw_edge_uniforms(obe):
    """u = 0 picks the first particle with weight, u -> 1 the last; zero-weight runs are skipped."""
    w = np.array([0, 0, .5, 0, .5, 0, 0], dtype=np.float64)
    pdf = obe.ParticlePDF(np.arange(7, dtype=np.float64).reshape(1, 7), resampling='multinomial')
    pdf.particle_weights = w

    class FixedRng:
        def __init__(self, vals):
            self.vals = np.asarray(vals)

        def random(self, n=None):
            return self.vals
    pdf.rng = FixedRng([0.0, 0.25, 0.5, np.nextafter(1.0, 0.0)])
    got = pdf.randdraw(4)[0]
    want = orc.choice_indices(w, pdf.rng.vals)
    assert_array_equal(got, want.astype(np.float64))


@pytest.mark.parametrize('scale', [True, False])
def test_multinomial_resample_matches_oracle(obe, scale):
    """Reference-parity resample: same Generator stream -> same ancestors (bit-exact) and the same
    Liu-West particles (particlepdf.py:286-310)."""
    n, d = 20000, 3
    rng = np.random.default_rng(4)
    prior = np.array([rng.uniform(2, 4, n), rng.uniform(-2000, -400, n), rng.normal(5e4, 1e3, n)])
    w = rng.random(n) ** 4
    w /= w.sum()
    pdf = obe.ParticlePDF(prior, scale=scale, resampling='multinomial')
    pdf.particle_weights = w
    pdf.rng = np.random.default_rng(99)
    g = np.random.default_rng(99)
    u, z = g.random(n), g.standard_normal(n * d)
    want, want_w, want_idx = orc.resample(prior, w, u, z, 0.98, scale)
    pdf.resample()
    assert_array_equal(pdf._last_ancestors.cpu().numpy(), want_idx)
    spread = prior.std(axis=1, keepdims=True)
    err = np.abs(pdf.particles - want) / (np.abs(want) * 1e-13 + spread * 1e-12)
    assert err.max() <= 1.0, err.max()
    assert_array_equal(pdf.particle_weights, want_w)
    assert pdf.rng.random() == g.random()                        # identical Generator state afterwards


@pytest.mark.parametrize('n,d', [(4096, 3), (10000, 3), (250001, 3), (1, 2), (2, 2), (5, 1), (2047, 2), (2049, 2),
                                 (4097, 1), (10000, 1), (30011, 4), (10000, 6), (6151, 8)])
@pytest.mark.parametrize('scale', [False, True])
@pytest.mark.parametrize('plan', ['one_cta', 'cluster'])
@pytest.mark.parametrize('kernel', ['warp_fused', 'two_kernel'])
def test_systematic_resample_matches_oracle(obe, torch, n, d, scale, plan, kernel):
    """Systematic resample (plan + the warp-autonomous fused kernel, or plan + ancestors + move): ancestors ==
    searchsorted(cdf_gpu, comb) bit-exact; normals are the restated Philox/Box-Muller stream; particles ==
    Liu-West with the Cholesky factor.  Sizes around the tile boundaries, every register variant of the kernels (d)."""
    from optbayesexpt_b200 import _lib
    # the resample plan on one CTA, or on the cluster of 8 CTAs that large clouds (> 8192 tiles) get
    _lib.check(_lib.load().obe_set_option(b'plan_cluster_min_tiles', 0 if plan == 'cluster' else 1 << 40))
    _lib.check(_lib.load().obe_set_option(b'resample_fused', 1 if kernel == 'warp_fused' else 0))
    try:
        _systematic_case(obe, torch, n, d, scale)
    finally:
        _lib.check(_lib.load().obe_set_option(b'plan_cluster_min_tiles', 8192))
        _lib.check(_lib.load().obe_set_option(b'resample_fused', 1))


@pytest.mark.parametrize('n,d,heavy', [(3_000_001, 3, False), (1_000_003, 2, True), (700_001, 5, False),
                                       (2_000_000, 1, True)])
def test_fused_resample_equals_two_kernel(obe, torch, n, d, heavy):
    """The one-kernel (warp-autonomous) systematic resample and the ancestors + move pair are the same function:
    identical ancestors, identical normals, bit-identical offspring -- at sizes with many work units per warp, with
    heavy particles that own many chunks of output slots, and with runs of dead particles."""
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator(device='cuda')
    g.manual_seed(n)
    prior = torch.randn((d, n), generator=g, dtype=torch.float64, device='cuda') * 3 + 1
    w = torch.rand(n, generator=g, dtype=torch.float64, device='cuda') ** 4
    w[torch.rand(n, generator=g, dtype=torch.float64, device='cuda') < 0.25] = 0.0
    if heavy:
        w[12345] = w.sum() * 0.3                                   # owns ~23 % of the slots: hundreds of chunks
        w[n - 7] = w.sum() * 0.05
        w[2048 * 100: 2048 * 140] = 0.0                            # forty dead tiles in a row
    w /= w.sum()
    out = {}
    for fused in (1, 0):
        pdf = obe.ParticlePDF(prior, scale=True, resampling='systematic', seed=5)
        pdf.particle_weights = w.cpu().numpy()
        pdf._ensure_moments()
        alt = pdf._buf.empty_like()
        idx = torch.empty(n, dtype=torch.int64, device='cuda')
        _lib.check(lib.obe_set_option(b'resample_fused', fused))
        try:
            _lib.check(lib.obe_resample_systematic(pdf._cs(), C.byref(alt.struct()), 0.61803, None, None, 42, 7, 0.98, 1,
                                                   C.c_void_p(idx.data_ptr()), None, pdf._stream()))
        finally:
            _lib.check(lib.obe_set_option(b'resample_fused', 1))
        out[fused] = (idx.clone(), alt.particles[:, :n].clone(), alt.stats.clone(), alt.tile_prefix.clone())
    assert torch.equal(out[1][0], out[0][0])
    assert torch.equal(out[1][1], out[0][1])
    assert torch.equal(out[1][2], out[0][2]) and torch.equal(out[1][3], out[0][3])
    idx = out[1][0]
    assert bool((idx[1:] >= idx[:-1]).all()) and int(idx[0]) >= 0 and int(idx[-1]) < n
    counts = torch.bincount(idx, minlength=n).to(torch.float64)
    assert float((counts - n * w).abs().max()) < 1.0 + 1e-6


def _systematic_case(obe, torch, n, d, scale):
    from optbayesexpt_b200 import _lib
    rng = np.random.default_rng(n)
    rows = [rng.uniform(2, 4, n), rng.uniform(-2000, -400, n), rng.normal(5e4, 1e3, n), rng.exponential(3.0, n),
            rng.normal(0, 1e-3, n), rng.uniform(-1, 1, n), rng.normal(7, 2, n), rng.uniform(0, 1e6, n)]
    prior = np.array(rows[:d])
    w = rng.random(n) ** 6
    w[rng.random(n) < 0.3] = 0.0                                  # runs of dead particles
    if w.sum() == 0.0:
        w[:] = 1.0
    w /= w.sum()
    pdf = obe.ParticlePDF(prior, scale=scale, resampling='systematic', seed=11)
    pdf.particle_weights = w
    lib = _lib.load()
    cdf = torch.empty(n, dtype=torch.float64, device='cuda')
    _lib.check(lib.obe_cdf(pdf._cs(), C.c_void_p(cdf.data_ptr()), pdf._stream()))
    cdf_h = cdf.cpu().numpy()
    pdf._ensure_moments()
    cov, mean = pdf.covariance(), pdf.mean()
    alt = pdf._buf.empty_like()
    idx = torch.empty(n, dtype=torch.int64, device='cuda')
    zout = torch.empty((n, d), dtype=torch.float64, device='cuda')
    u0, seed, epoch = 0.37, 123456789, 3
    _lib.check(lib.obe_resample_systematic(pdf._cs(), C.byref(alt.struct()), u0, None, None, seed, epoch, 0.98,
                                           1 if scale else 0, C.c_void_p(idx.data_ptr()),
                                           C.c_void_p(zout.data_ptr()), pdf._stream()))
    idx_h = idx.cpu().numpy()
    want_idx = orc.search_cdf(cdf_h, orc.systematic_uniforms(u0, n))
    assert_array_equal(idx_h, want_idx)
    # offspring counts of systematic resampling: floor(n w) or ceil(n w) (up to CDF rounding)
    counts = np.bincount(idx_h, minlength=n)
    assert np.all(np.abs(counts - n * w) < 1.0 + 1e-6)
    # the normals: the restated Philox + float32 Box-Muller stream, to float32 accuracy; the
    # Liu-West arithmetic downstream is then checked exactly, GIVEN the normals the kernel used
    z = zout.cpu().numpy()
    assert_allclose(z, orc.device_normals_packed(n, d, seed, epoch), rtol=0, atol=1e-4)
    if n * d >= 1000:
        assert abs(z.mean()) < 5 / np.sqrt(n * d) and abs(z.std() - 1) < 5 / np.sqrt(n * d)
    if n < 3:
        return                                                    # no covariance to speak of
    f = orc.mvn_factor_cholesky((1 - 0.98 ** 2) * np.atleast_2d(cov))
    want = orc.liu_west(prior[:, want_idx], z, f, 0.98, scale, mean)
    got = alt.particles[:, :n].cpu().numpy()
    spread = prior.std(axis=1, keepdims=True)
    err = np.abs(got - want) / (np.abs(want) * 1e-13 + spread * 1e-11)
    assert err.max() <= 1.0, err.max()
    # the offspring weights are implicit (never written) until something asks for the row
    assert float(alt.stats[62].item()) == 1.0 / n
    _lib.check(lib.obe_materialize_weights(C.byref(alt.struct()), pdf._stream()))
    assert float(alt.stats[62].item()) == 0.0
    assert_array_equal(alt.weights[:n].cpu().numpy(), np.full(n, 1.0 / n))


def test_systematic_extreme_weights(obe, torch):
    """One particle owns (almost) everything; another cloud has a single survivor per tile."""
    n = 3 * 2048 + 17
    prior = np.arange(n, dtype=np.float64).reshape(1, n)
    w = np.full(n, 1e-30)
    w[4000] = 1.0
    w /= w.sum()
    pdf = obe.ParticlePDF(prior, scale=False, resampling='systematic', seed=1)
    pdf.tuning_parameters['a_param'] = 1.0                       # no jitter: children are exact copies
    pdf.particle_weights = w
    pdf.resample()
    assert_array_equal(pdf.particles[0], np.full(n, 4000.0))
    w = np.zeros(n)
    w[[5, 2048 + 7, 2 * 2048 + 9, n - 1]] = 0.25
    pdf = obe.ParticlePDF(prior, scale=False, resampling='systematic', seed=1)
    pdf.tuning_parameters['a_param'] = 1.0
    pdf.particle_weights = w
    pdf.resample()
    vals, counts = np.unique(pdf.particles[0], return_counts=True)
    assert_array_equal(vals, [5, 2048 + 7, 2 * 2048 + 9, n - 1])
    assert counts.sum() == n and np.all(np.abs(counts - n / 4) <= 1)


@pytest.mark.parametrize('name', ['c1_find_peak', 'c2_line_noise', 'c3_pipulse', 'c5_lockin'])
def test_utility_and_selection_match_oracle(obe, name):
    sc = by_name(name)
    eng, inp = _engine(obe, sc)
    eng.tuning_parameters['auto_resample'] = False
    rec = RECORDS[name]
    if sc['kind'] != 'base':
        rec = (rec[0], rec[1], None)
    eng.pdf_update(rec)
    w = eng.particle_weights
    model, _, _, _, nch = orc.MODELS[sc['model']]
    g = np.random.default_rng(31)
    eng.rng = np.random.default_rng(31)
    draws, _ = orc.randdraw(inp['prior'], np.asarray(w), g.random(sc['n_draws']))
    var_p, _ = orc.yvar_from_draws(model, orc.make_allsettings(inp['setting_values']), draws, inp['cons'], nch)
    if sc['kind'] == 'base':
        var_n = orc.noise_var_default(sc.get('default_noise_std', 1.0), nch)
    else:
        var_n = orc.noise_var_noise_parameter(inp['prior'], np.asarray(w), sc['noise_parameter_index'])
    cost = 1.0
    if sc['kind'] == 'lockin':
        cost = orc.lockin_cost(var_p.shape[1], 0, sc['cost_of_changing_setting'])
    want_u = orc.utility_variance(var_p, var_n, cost)
    got = eng.opt_setting()
    got_u = eng._utility_dev.cpu().numpy()
    assert_allclose(got_u, want_u, rtol=1e-12)
    assert eng.last_setting_index == orc.opt_index(want_u)
    assert got == tuple(orc.make_allsettings(inp['setting_values'])[:, orc.opt_index(want_u)])
    # pickiness-weighted draw (obe_base.py:778-789) with the same uniform
    eng.rng = np.random.default_rng(32)
    g = np.random.default_rng(32)
    draws, _ = orc.randdraw(inp['prior'], np.asarray(w), g.random(sc['n_draws']))
    var_p, _ = orc.yvar_from_draws(model, orc.make_allsettings(inp['setting_values']), draws, inp['cons'], nch)
    if sc['kind'] == 'lockin':
        cost = orc.lockin_cost(var_p.shape[1], eng.last_setting_index, sc['cost_of_changing_setting'])
    want_u = orc.utility_variance(var_p, var_n, cost)
    eng.good_setting(pickiness=4)
    assert eng.last_setting_index == orc.good_index(want_u, 4, g.random())


def test_rational_model_utility_is_bit_exact(obe):
    """Lorentzian / line use non-contracted IEEE ops in numpy's order: the utility must agree to the
    last bit, so the argmax can never flip."""
    sc = by_name('c1_find_peak')
    eng, inp = _engine(obe, sc)
    eng.rng = np.random.default_rng(8)
    g = np.random.default_rng(8)
    w = np.ones(sc['n_particles']) / sc['n_particles']
    draws, _ = orc.randdraw(inp['prior'], w, g.random(30))
    var_p, _ = orc.yvar_from_draws(orc.model_lorentzian_hwhm, orc.make_allsettings(inp['setting_values']), draws,
                                   inp['cons'], 1)
    want = orc.utility_variance(var_p, orc.noise_var_default(500.0, 1))
    assert_array_equal(eng.utility(), want)


def test_argmax_ties_pick_lowest_index(obe):
    """Duplicate settings (tests/test_server.py:26 uses [0,1,0]) -> first maximum, like np.argmax."""
    prior = np.array([np.linspace(-1, 1, 4096), np.linspace(0.5, 2, 4096)])
    eng = obe.OptBayesExpt('line', (np.array([1.0, 0.0, 1.0, 0.5, 1.0] * 1000),), prior, (), seed=3)
    eng.opt_setting()
    util = eng._utility_dev.cpu().numpy()
    assert eng.last_setting_index == int(np.argmax(util)) == 0


def test_max_min_and_log_utility(obe):
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc)
    eng = obe.OptBayesExpt('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons'],
                           utility_method='max_min', default_noise_std=500.0)
    eng.rng = np.random.default_rng(8)
    g = np.random.default_rng(8)
    w = np.ones(sc['n_particles']) / sc['n_particles']
    draws, _ = orc.randdraw(inp['prior'], w, g.random(30))
    _, ys = orc.yvar_from_draws(orc.model_lorentzian_hwhm, orc.make_allsettings(inp['setting_values']), draws,
                                inp['cons'], 1)
    span2 = (ys.max(axis=0) - ys.min(axis=0)) ** 2             # obe_base.py:532-535
    assert_allclose(eng.utility(), np.sum(span2 / 500.0 ** 2, axis=0), rtol=1e-14)
    eng2 = obe.OptBayesExpt('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons'],
                            default_noise_std=500.0)
    eng2.utility_log_form = True
    eng2.rng = np.random.default_rng(8)
    var_p = np.var(ys, axis=0)
    assert_allclose(eng2.utility(), orc.utility_variance(var_p, 500.0 ** 2, 1.0, log_form=True), rtol=1e-13)


def test_device_model_call_both_orientations(obe):
    """DeviceModel keeps the reference's broadcasting contract (obe_base.py:50-66), on the GPU."""
    m = obe.builtin('lorentzian_hwhm')
    x = np.linspace(1.5, 4.5, 77)
    assert_array_equal(m((x,), (3.0, -1000.0, 5e4), (0.1,)),
                       orc.model_lorentzian_hwhm((x,), (3.0, -1000.0, 5e4), (0.1,)))
    rng = np.random.default_rng(0)
    pars = (rng.uniform(2, 4, 501), rng.uniform(-2000, -400, 501), rng.normal(5e4, 1e3, 501))
    assert_array_equal(m((2.5,), pars, (0.1,)), orc.model_lorentzian_hwhm((2.5,), pars, (0.1,)))
    assert m((2.5,), (3.0, -1000.0, 5e4), (0.1,)) == orc.model_lorentzian_hwhm((2.5,), (3.0, -1000.0, 5e4), (0.1,))
    lock = obe.builtin('lockin_coil')
    wv = 2 * np.pi * np.logspace(2, 6, 50)
    assert_allclose(lock((wv,), (1.2e-3, 8.0, 0.9e-5), ()), orc.model_lockin_coil((wv,), (1.2e-3, 8.0, 0.9e-5), ()),
                    rtol=1e-14)
    rabi = obe.builtin('rabi')
    tt, ff = np.meshgrid(np.linspace(0, 1, 11), np.linspace(-10, 10, 11), indexing='ij')
    assert_allclose(rabi((tt, ff), (3.3, 1.7), (1e5, 0.01, 0.5)), orc.model_rabi((tt, ff), (3.3, 1.7), (1e5, 0.01, 0.5)),
                    rtol=1e-14)


def test_nvrtc_user_model_equals_builtin(obe):
    src = '''
    __device__ void my_lorentz(const double* s, const double* p, const double* c, double* y) {
        const double q = obe_div(obe_sub(s[0], p[0]), c[0]);
        y[0] = obe_add(p[2], obe_div(p[1], obe_add(obe_mul(q, q), 1.0)));
    }'''
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc)
    user = obe.cuda_source(src, 'my_lorentz', n_settings=1, n_params=3, n_constants=1)
    a = obe.OptBayesExpt(user, inp['setting_values'], inp['prior'], inp['cons'], seed=5, default_noise_std=500.0)
    b = obe.OptBayesExpt('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons'], seed=5,
                         default_noise_std=500.0)
    for eng in (a, b):
        eng.tuning_parameters['auto_resample'] = False
    assert a.opt_setting() == b.opt_setting()
    a.pdf_update(RECORDS['c1_find_peak'])
    b.pdf_update(RECORDS['c1_find_peak'])
    # the built-in's update pass hoists 1/d out of the loop; the user functor divides: last-bit differences
    wclose(a.particle_weights, b.particle_weights, 1e-12)
    bad = obe.cuda_source('__device__ void broken(', 'broken', 1, 3)
    from optbayesexpt_b200._lib import ObeError
    with pytest.raises(ObeError):
        bad.handle(3)


# =================================================================================================
# 3. closed-loop golden trajectories of the unmodified reference
# =================================================================================================
@pytest.mark.parametrize('sc', SCENARIOS, ids=[s['name'] for s in SCENARIOS])
def test_golden_trajectory(obe, sc):
    """Seeded exactly like the reference run that wrote the golden file: every chosen setting index
    and every resample decision must be identical; utility / moments / weights within the
    (condition-aware) tolerance."""
    g = np.load(os.path.join(GOLDEN, sc['name'] + '.npz'))
    eng, inp = _engine(obe, sc, pickiness=sc.get('pickiness', 15))
    nch = orc.MODELS[sc['model']][4]
    tol = sc.get('traj_rtol', 1e-9)
    cols = g['utility_columns'] if 'utility_columns' in g.files else slice(None)   # (a large grid is sampled)
    seen = False
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for t in range(sc['n_cycles']):
            setting = eng.good_setting() if sc['selection'] == 'good' else eng.opt_setting()
            assert eng.last_setting_index == g['set_index'][t], f'setting index differs at cycle {t}'
            assert_allclose(eng._utility_dev.cpu().numpy()[cols], g['utility'][t], rtol=tol if seen else 1e-12,
                            err_msg=f'utility t={t}')
            y, sig = g['y_meas'][t], g['sigma_meas'][t]
            rec = (setting, tuple(y) if nch > 1 else float(y[0]), tuple(sig) if nch > 1 else float(sig[0]))
            eng.pdf_update(rec)
            assert int(eng.just_resampled) == g['resampled'][t], f'resample decision differs at cycle {t}'
            if eng.just_resampled and not seen:
                assert_array_equal(eng._last_ancestors.cpu().numpy(), g['first_ancestors'])
            seen = seen or eng.just_resampled
            assert_allclose(eng.mean(), g['mean'][t], rtol=tol if seen else 1e-12, err_msg=f'mean t={t}')
            cov_close(eng.covariance(), g['cov'][t], max(tol, 1e-9))
    wclose(eng.particle_weights, g['final_weights'], max(tol, 1e-9))
    spread = g['final_particles'].std(axis=1, keepdims=True)
    err = np.abs(eng.particles - g['final_particles']) / (np.abs(g['final_particles']) * 1e-9 + spread * 1e-8)
    assert err.max() <= 1.0


def test_closed_loop_systematic_converges(obe):
    """Default (systematic, device RNG) engine on config c1: no golden for it, so check the physics --
    the posterior mean lands on the truth within a few posterior sigmas."""
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc)
    eng = obe.OptBayesExpt('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons'], scale=False,
                           default_noise_std=500.0, seed=21)
    meas = np.random.default_rng(22)
    n_res = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(150):
            s = eng.opt_setting()
            y = orc.model_lorentzian_hwhm(s, sc['true_pars'], inp['cons']) + 500.0 * meas.standard_normal()
            eng.pdf_update((s, float(y), 500.0))
            n_res += int(eng.just_resampled)
    assert n_res > 0
    err = np.abs(eng.mean() - np.array(sc['true_pars'])) / eng.std()
    assert np.all(err < 5), (eng.mean(), eng.std())
    assert eng.std()[0] < 0.01


# =================================================================================================
# 4. size-independent properties at the BASELINE scale (N = 1e8 would not finish on the oracle)
# =================================================================================================
def test_full_scale_properties(obe, torch):
    n = 20_000_000
    gen = torch.Generator(device='cuda')
    gen.manual_seed(1001)
    prior = torch.empty((3, n), dtype=torch.float64, device='cuda')
    prior[0] = 2 + 2 * torch.rand(n, generator=gen, dtype=torch.float64, device='cuda')
    prior[1] = -2000 + 1600 * torch.rand(n, generator=gen, dtype=torch.float64, device='cuda')
    prior[2] = 50000 + 1000 * torch.randn(n, generator=gen, dtype=torch.float64, device='cuda')
    eng = obe.OptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 100000),), prior, (0.1,), scale=False,
                           default_noise_std=500.0, seed=7)
    eng.tuning_parameters['auto_resample'] = False
    eng.pdf_update(((3.1,), 49600.0, 500.0))
    w = eng.weights_dev * eng.weight_scale
    assert abs(float(w.sum()) - 1.0) < 1e-12
    # the same N_eff from an independent torch reduction
    assert_allclose(eng.n_eff(), 1.0 / float((w * w).sum()), rtol=1e-11)
    mean_t = (eng.particles_dev * w).sum(dim=1).cpu().numpy()
    assert_allclose(eng.mean(), mean_t, rtol=1e-11)
    # prefix of tile sums is a CDF: monotone, ends at the total
    pre = eng._buf.tile_prefix.cpu().numpy()
    assert np.all(np.diff(pre) >= 0)
    assert_allclose(pre[-1], float(eng.weights_dev.sum()), rtol=1e-12)
    before_mean, before_cov = eng.mean(), eng.covariance()
    eng.resample()
    # resampling refreshes the representation, it must not move the distribution (Liu-West with
    # scale=False inflates the covariance by exactly 1 + (1 - a^2))
    assert_array_equal(eng.weights_dev.cpu().numpy()[:1000], np.full(1000, 1.0 / n))
    sd = np.sqrt(np.diag(before_cov))
    assert np.all(np.abs(eng.mean() - before_mean) < 5 * sd / np.sqrt(eng.n_eff() if False else 1e6))
    ratio = np.diag(eng.covariance()) / np.diag(before_cov)
    assert_allclose(ratio, 1 + (1 - 0.98 ** 2), rtol=5e-3)
    s = eng.opt_setting()
    assert 1.5 <= s[0] <= 4.5


# =================================================================================================
# 5. the remaining utility methods (SURVEY 8f "next" row 1): pseudo-utility and full KLD
# =================================================================================================
@pytest.mark.parametrize('n_draws', [8, 30, 100])      # van Es (n <= 10) and Ebrahimi estimators
def test_pseudo_utility_matches_oracle(obe, n_draws):
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc)
    eng = obe.OptBayesExpt('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons'],
                           utility_method='pseudo_utility', default_noise_std=500.0, n_draws=n_draws)
    eng.rng = np.random.default_rng(17)
    g = np.random.default_rng(17)
    w = np.ones(sc['n_particles']) / sc['n_particles']
    draws, _ = orc.randdraw(inp['prior'], w, g.random(n_draws))
    _, ys = orc.yvar_from_draws(orc.model_lorentzian_hwhm, orc.make_allsettings(inp['setting_values']), draws,
                                inp['cons'], 1)
    want = orc.utility_pseudo(ys, orc.noise_var_default(500.0, 1))
    got = eng.utility()
    assert_allclose(got, want, rtol=1e-12)
    eng.rng = np.random.default_rng(17)
    eng.opt_setting()
    assert eng.last_setting_index == orc.opt_index(want)


def test_pseudo_utility_two_channels(obe):
    sc = by_name('c5_lockin')
    inp = build_inputs(sc)
    eng = obe.OptBayesExptNoiseParameter('lockin_coil', inp['setting_values'], inp['prior'], inp['cons'],
                                         noise_parameter_index=(3, 3), utility_method='pseudo_utility')
    eng.rng = np.random.default_rng(3)
    g = np.random.default_rng(3)
    w = np.ones(sc['n_particles']) / sc['n_particles']
    draws, _ = orc.randdraw(inp['prior'], w, g.random(30))
    _, ys = orc.yvar_from_draws(orc.model_lockin_coil, orc.make_allsettings(inp['setting_values']), draws, (), 2)
    want = orc.utility_pseudo(ys, orc.noise_var_noise_parameter(inp['prior'], w, (3, 3)))
    assert_allclose(eng.utility(), want, rtol=1e-11)


def test_full_kld_utility_matches_oracle(obe):
    import optbayesexpt_b200.obe_base as base
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc)
    eng = obe.OptBayesExpt('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons'],
                           utility_method='full_kld_utility', default_noise_std=500.0)
    eng.rng = np.random.default_rng(17)
    base.rng = np.random.default_rng(23)                    # the reference's module-level Generator
    g = np.random.default_rng(17)
    w = np.ones(sc['n_particles']) / sc['n_particles']
    draws, _ = orc.randdraw(inp['prior'], w, g.random(30))
    _, ys = orc.yvar_from_draws(orc.model_lorentzian_hwhm, orc.make_allsettings(inp['setting_values']), draws,
                                inp['cons'], 1)
    nva = np.random.default_rng(23).normal(0, 1.0, 30).reshape((1, 30))
    noise = (nva * np.sqrt(orc.noise_var_default(500.0, 1))).T
    want = orc.utility_full_kld(ys, noise)[0]
    got = eng.utility()
    assert_allclose(got, want, rtol=1e-11)
    with pytest.raises(ValueError):
        obe.OptBayesExptNoiseParameter('lockin_coil', (np.linspace(1, 2, 5),), np.ones((4, 64)), (),
                                       noise_parameter_index=(3, 3), utility_method='full_kld_utility')
