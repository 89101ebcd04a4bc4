"""The batched engines' random-walk drift on the device: the pass against the oracle's keying and numpy's moments, what
it must leave alone, instance independence, zero drift, the constraint masks, the default path, the covariance it
adds, the simulator's truth walk, a closed loop that tracks drifting peaks, the setter, and the C-level refusals."""
import ctypes as C
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from oracle import batched_drift as obd
from oracle import drift as odr
from oracle import obe_oracle as orc
from oracle.scenarios import build_inputs, by_name

pytestmark = pytest.mark.gpu

# a one-parameter model: the cloud may have any number of rows (1 .. 8) behind it
LINE_SRC = '__device__ void slope(const double* s, const double* p, const double* c, double* y) { y[0] = p[0] * s[0]; }\n'


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


def _np(t):
    return t.detach().cpu().numpy().copy()


_SLOPE = []


def _slope_engine(obe, prior, seed=7, **kw):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    from optbayesexpt_b200.models import cuda_source
    if not _SLOPE:
        _SLOPE.append(cuda_source(LINE_SRC, 'slope', 1, 1))         # (one NVRTC compile per n_params)
    return BatchedOptBayesExpt(_SLOPE[0], (np.linspace(0.0, 1.0, 5),), prior, (), scale=False, seed=seed,
                               default_noise_std=1.0, **kw)


def _random_weights(beng, g):
    """Explicit non-uniform weights in the live slots, then the refresh passes that rebuild every derived quantity."""
    import torch
    from optbayesexpt_b200 import _lib
    w = np.zeros((beng.n_instances, beng._np))
    w[:, :beng.n_particles] = g.uniform(0.05, 1.0, (beng.n_instances, beng.n_particles))
    beng._w[0].copy_(torch.from_numpy(w.reshape(-1)))
    for _ in range(2):
        beng._check(beng._lib.obe_batch_refresh(beng._bs(), 0, 0, None, 0, beng._stream()))
    torch.cuda.synchronize()
    assert _lib.ST_TOTAL == 0


def _snapshot(beng):
    import torch
    torch.cuda.synchronize()
    names = ('_cur', '_tile_sums', '_prefix', '_stats', '_pivot', '_record', '_last_idx', '_flag', '_epoch')
    snap = {k: _np(getattr(beng, k)) for k in names}
    snap['p0'], snap['p1'] = _np(beng._p[0]), _np(beng._p[1])
    snap['w0'], snap['w1'] = _np(beng._w[0]), _np(beng._w[1])
    return snap


def _factor(g, d, zero_row=True):
    from optbayesexpt_b200.drift import drift_factor
    a = g.normal(size=(d, d)) * 0.05
    q = a @ a.T
    if zero_row and d > 1:
        q[d // 2, :] = q[:, d // 2] = 0.0
    return drift_factor(q, d)


def _pass(beng, shared, per, seed, step, mask_le=0, mask_lt=0):
    from optbayesexpt_b200 import _lib
    dev = None if per is None else beng._to_device(per)
    beng._check(beng._lib.obe_batch_drift(beng._bs(), None if shared is None else _lib.darr(shared.reshape(-1)),
                                          beng._ptr(dev), mask_le, mask_lt, None, 0, seed, step, beng._stream()))
    import torch
    torch.cuda.synchronize()


def _check_moved(x, after, factor, z):
    """after = x + F z to the float32 accuracy of the device normals (see test_gpu_drift.py: |dz| < 1e-3 always,
    < 1e-5 but for ~1e-4 of them)."""
    want = x + factor @ z.T
    scale = np.abs(factor).sum(axis=1)[:, None]
    err = np.abs(after - want) - 1e-12 * np.abs(want)
    assert np.all(err <= 1e-3 * scale)
    assert np.mean(err > 1e-5 * scale) < 2e-4


UNCHANGED_STATS = ('ST_TOTAL', 'ST_INVS', 'ST_SUMSQ', 'ST_NEFF', 'ST_SUMT', 'ST_NZERO', 'ST_UNIFORM', 'ST_FIRED')


@pytest.mark.parametrize('per_instance', [False, True])
@pytest.mark.parametrize('d', [1, 4, 8])
@pytest.mark.parametrize('n', [1000, 10_000, 131_072])
def test_pass_parity(obe, n, d, per_instance):
    from optbayesexpt_b200 import _lib
    B, seed, step = 64, 0x1234567890ABCDEF, 11
    g = np.random.default_rng(n + d)
    prior = g.normal(size=(B, d, n)) + np.arange(1, d + 1)[None, :, None]
    beng = _slope_engine(obe, prior)
    _random_weights(beng, g)
    if per_instance:
        factors = np.stack([_factor(g, d, zero_row=(b % 3 == 0)) for b in range(B)])
        factors[5] = 0.0                                   # an instance that does not drift
        shared = None
    else:
        shared = _factor(g, d)
        factors = np.broadcast_to(shared, (B, d, d))
    before = _snapshot(beng)
    _pass(beng, shared, factors if per_instance else None, seed, step)
    after = _snapshot(beng)
    # everything but the live particle rows and the moments: bit for bit
    for key in ('p1', 'w0', 'w1', '_cur', '_tile_sums', '_prefix', '_record', '_last_idx', '_flag', '_epoch'):
        assert_array_equal(after[key], before[key], err_msg=key)
    same = [getattr(_lib, s) for s in UNCHANGED_STATS]
    assert_array_equal(after['_stats'][:, same], before['_stats'][:, same])
    npad = beng._np
    p_before = before['p0'].reshape(d, B, npad)
    p_after = after['p0'].reshape(d, B, npad)
    assert_array_equal(p_after[:, :, n:], p_before[:, :, n:])      # padding slots
    # the moved rows against the oracle's keying, on a sample of instances
    for b in (0, 5, 33, B - 1):
        x, moved = p_before[:, b, :n], p_after[:, b, :n]
        z = obd.batched_drift_normals(n, d, seed, step, b)
        _check_moved(x, moved, factors[b], z)
        for j in range(d):
            if np.all(factors[b][j] == 0.0):
                assert_array_equal(moved[j], x[j])
    # the moments of every instance against numpy on the downloaded cloud
    w = before['w0'].reshape(B, npad)[:, :n]
    st = after['_stats']
    for b in range(B):
        piv = before['_pivot'][b, :d]
        assert_array_equal(st[b, _lib.ST_PIVOT:_lib.ST_PIVOT + d], piv)
        dx = p_after[:, b, :n] - piv[:, None]
        m1 = (w[b] * dx).sum(axis=1)
        assert_allclose(st[b, _lib.ST_M1:_lib.ST_M1 + d], m1, rtol=1e-12,
                        atol=1e-12 * np.abs(w[b] * dx).sum(axis=1).max())
        q = _lib.ST_M2
        for j in range(d):
            for k in range(j, d):
                terms = w[b] * dx[j] * dx[k]
                assert_allclose(st[b, q], terms.sum(), rtol=1e-12, atol=1e-12 * np.abs(terms).sum())
                q += 1
        # the next pass's pivot: the drifted mean
        assert_allclose(after['_pivot'][b, :d], piv + m1 / w[b].sum(), rtol=1e-10, atol=1e-12)


def test_instances_are_independent(obe):
    """Instance b's rows and stats after a pass are the same bits with 8 or 64 instances, whatever the other
    instances' factors are."""
    n, d = 10_000, 4
    g = np.random.default_rng(3)
    prior = g.normal(size=(64, d, n))
    qs = []
    for b in range(64):
        a = g.normal(size=(d, d)) * 0.03
        qs.append(a @ a.T)
    qs = np.stack(qs)
    qs_other = qs.copy()
    qs_other[8:] *= 7.0
    out = []
    for B, q in ((8, qs[:8]), (64, qs), (64, qs_other)):
        beng = _slope_engine(obe, prior[:B], seed=9, drift=q)
        for _ in range(3):
            beng._apply_drift()
        s = _snapshot(beng)
        out.append((s['p0'].reshape(d, B, beng._np)[:, :8], s['_stats'][:8], s['_pivot'][:8]))
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert_array_equal(a, b)


def test_zero_drift_keeps_the_bits(obe):
    n, d, B = 5000, 3, 6
    g = np.random.default_rng(4)
    prior = g.normal(size=(B, d, n))
    beng = _slope_engine(obe, prior, drift=np.zeros((d, d)))
    x = _snapshot(beng)['p0']
    beng._apply_drift()
    assert_array_equal(_snapshot(beng)['p0'], x)
    # zero-variance rows of per-instance covariances
    qs = np.stack([np.diag([0.01, 0.02, 0.03])] * B)
    qs[2] = 0.0
    qs[4][1, :] = qs[4][:, 1] = 0.0
    beng.drift = qs
    beng._apply_drift()
    y = _snapshot(beng)['p0'].reshape(d, B, beng._np)
    x = x.reshape(d, B, beng._np)
    assert_array_equal(y[:, 2], x[:, 2])
    assert_array_equal(y[1, 4], x[1, 4])
    assert not np.any(y[0, 4, :n] == x[0, 4, :n])


def _lockin_engine(obe, B, n, seed=11, **kw):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    sc = by_name('c5_lockin')
    inp = build_inputs(sc, n)
    rng = np.random.default_rng(seed)
    prior = np.stack([sc['prior'](rng, n) for _ in range(B)])
    beng = BatchedOptBayesExpt('lockin_coil', inp['setting_values'], prior, (), noise_parameter_index=(3, 3),
                               constraint_lt=(0, 1, 2, 3), cost_of_changing_setting=5.0, scale=False, seed=seed, **kw)
    return beng, sc, prior


def test_masks_keep_the_noise_parameter_positive(obe):
    B, n = 16, 10_000
    beng, sc, prior = _lockin_engine(obe, B, n)
    # steps of the noise parameter as large as its typical value: many would cross zero
    scale = np.median(prior[:, 3])
    drift = [0.0, 0.0, 0.0, scale]
    beng.drift = drift
    x = _snapshot(beng)['p0'].reshape(4, B, beng._np)[:, :, :n]
    beng._apply_drift()
    y = _snapshot(beng)['p0'].reshape(4, B, beng._np)[:, :, :n]
    for b in (0, 7, 15):
        z = obd.batched_drift_normals(n, 4, beng._seed_normal, beng._drift_step, b)
        want, ok = odr.drift_step(x[:, b], np.diag(drift), z, mask_lt=0b1111)
        assert 0.05 < np.mean(~ok) < 0.95
        assert_array_equal(y[:, b, ~ok], x[:, b, ~ok])
        assert_allclose(y[:, b, ok], want[:, ok], rtol=1e-5, atol=1e-3 * scale)
    assert np.all(y[3] > 0.0)
    # and through closed-loop cycles on the device
    beng.set_simulator(np.tile(sc['true_pars'], (B, 1)), 5.0, seed=3)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(20):
            beng.closed_loop_cycle()
    # (the resample's jitter may still propose offspring outside the region: they get weight 0, as without drift;
    # the drift never takes a particle out of it, so every particle that carries weight is inside)
    for b in range(B):
        live = beng.particle_weights(b) > 0.0
        assert live.sum() > n // 10
        assert np.all(beng.particles(b)[3][live] > 0.0)
    assert np.all(np.isfinite(beng.mean()))


def test_default_path_is_unchanged(obe):
    B, n = 64, 10_000
    truths = np.tile(by_name('c5_lockin')['true_pars'], (B, 1))
    engines = []
    for kw in ({}, dict(drift=None)):
        beng, _, _ = _lockin_engine(obe, B, n, **kw)
        beng.set_simulator(truths, 5.0, seed=5)
        engines.append(beng)
    a, b = engines
    fired = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(50):
            a.closed_loop_cycle()
            b.closed_loop_cycle()
            fired += int(a.just_resampled.sum())
    assert fired > 0
    sa, sb = _snapshot(a), _snapshot(b)
    for key in sa:
        assert_array_equal(sa[key], sb[key], err_msg=key)
    assert a._drift_step == b._drift_step == 0


def test_covariance_grows_by_q(obe):
    """Uninformative records keep the weights uniform; every update adds Q to every instance's covariance (a full
    Q with correlations: F^T F in place of F F^T would fail)."""
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    B, n, cycles = 8, 131_072, 20
    g = np.random.default_rng(8)
    prior = g.normal(size=(B, 3, n)) * 0.05 + np.array([3.0, 1.0, -2.0])[None, :, None]
    q = np.array([[0.010, 0.006, -0.003], [0.006, 0.008, 0.002], [-0.003, 0.002, 0.005]])
    beng = BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 50),), prior, (0.1,), seed=3, drift=q)
    c0 = beng.covariance()
    for _ in range(cycles):
        beng.pdf_update(np.zeros((B, 1)), sigma=1e12, settings=np.full((B, 1), 3.0))
        assert not beng.just_resampled.any()
    grown = beng.covariance() - c0
    total = c0[0] + cycles * q
    tol = 6.0 * np.sqrt(np.outer(np.diag(total), np.diag(total)) * 2.0 / n)
    for b in range(B):
        assert np.all(np.abs(grown[b] - cycles * q) < tol), (b, grown[b], cycles * q, tol)
        assert_allclose(beng.mean()[b], beng.particles(b).mean(axis=1), rtol=1e-9)


def test_simulator_truth_walk(obe):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    from optbayesexpt_b200.drift import drift_factor
    sc = by_name('c1_find_peak')
    B, n, steps, seed = 4096, 2048, 40, 99
    inp = build_inputs(sc, n)
    g = np.random.default_rng(5)
    prior = np.broadcast_to(sc['prior'](g, n), (B, 3, n))
    beng = BatchedOptBayesExpt('lorentzian_hwhm', inp['setting_values'], prior, inp['cons'], scale=False,
                               default_noise_std=500.0, seed=4)
    truth0 = np.stack([g.uniform(2.2, 3.8, B), g.uniform(-1800, -600, B), g.normal(50000, 500, B)], axis=1)
    q = np.array([[1e-4, 2e-3, 0.0], [2e-3, 0.25, 0.1], [0.0, 0.1, 4.0]])
    beng.set_simulator(truth0, 500.0, seed=seed, drift=q)
    assert_array_equal(beng.simulator_truth(), truth0)
    f = drift_factor(q, 3)
    for t in range(steps):
        rec = beng.simulate_measurement().cpu().numpy()
        if t in (0, 7):
            # measurement t sees the truth after t steps
            settings = beng.allsettings[:, beng.last_setting_index]
            want = orc.simulate_batch_measurement(orc.model_lorentzian_hwhm, settings.T,
                                                  obd.truth_walk(truth0, f, seed, t), inp['cons'], 500.0, seed,
                                                  beng.cycle, 1)
            assert_allclose(rec[:, 4], want[:, 0], rtol=0, atol=500.0 * 1e-5)
    truth = beng.simulator_truth()
    want = obd.truth_walk(truth0, f, seed, steps)
    # float32 normals (see _check_moved): a rare |dz| up to 1e-3, ~1e-6 typically
    row = np.abs(f).sum(axis=1)
    err = np.abs(truth - want) - 1e-12 * np.abs(want)
    assert np.all(err <= 2e-3 * row) and np.all(np.median(err, axis=0) <= 1e-5 * row)
    step_cov = np.cov((truth - truth0).T)
    tol = 6.0 * np.sqrt(np.outer(np.diag(q), np.diag(q)) * 2.0 / B) * steps
    assert np.all(np.abs(step_cov - steps * q) < tol), (step_cov, steps * q)
    # per-instance truth covariances: instance b walks with its own F; zero rows keep their bits
    qs = np.stack([q * (1 + b % 4) for b in range(B)])
    qs[3] = 0.0
    beng.set_simulator(truth0, 500.0, seed=seed + 1, drift=qs)
    for _ in range(3):
        beng.simulate_measurement()
    fs = np.stack([drift_factor(x, 3) for x in qs])
    truth = beng.simulator_truth()
    want = obd.truth_walk(truth0, fs, seed + 1, 3)
    err = np.abs(truth - want) - 1e-12 * np.abs(want)
    assert np.all(err <= 2e-3 * np.abs(fs).sum(axis=2))
    assert_array_equal(truth[3], truth0[3])


def _tracking_errors(obe, drift, cycles=300, B=256, n=10_000, step=0.004):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    settings = (np.linspace(1.5, 4.5, 200),)
    g = np.random.default_rng(22)
    prior = np.stack([np.array([g.uniform(2, 4, n), g.uniform(-2000, -400, n), g.normal(50000, 1000, n)])
                      for _ in range(B)])
    beng = BatchedOptBayesExpt('lorentzian_hwhm', settings, prior, (0.1,), scale=False, default_noise_std=100.0,
                               seed=23, drift=drift)
    truths = np.stack([g.uniform(2.7, 3.3, B), np.full(B, -1200.0), np.full(B, 50400.0)], axis=1)
    beng.set_simulator(truths, 100.0, seed=24, drift=[step, 0.0, 0.0])
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        for _ in range(cycles):
            beng.closed_loop_cycle()
    # after the cycle the cloud and the truth both describe the next measurement
    return np.abs(beng.mean()[:, 0] - beng.simulator_truth()[:, 0]) / beng.std()[:, 0]


def test_matched_drift_tracks_drifting_peaks(obe):
    """256 Lorentzian peaks whose centres take a Gaussian random walk, in a closed loop on the device: with the
    matched drift the estimates stay within a few std of the truth; without drift the clouds collapse and lose it."""
    matched = _tracking_errors(obe, [0.004, 0.0, 0.0])
    static = _tracking_errors(obe, None)
    print('median |mean - truth| / std: matched', np.median(matched), 'static', np.median(static))
    assert np.median(matched) < 1.5, np.sort(matched)
    assert np.mean(matched < 4.0) > 0.9
    assert np.median(static) > 20.0, np.sort(static)


def test_setter_takes_effect_at_the_next_update(obe):
    n, d, B, seed = 4096, 3, 4, 31
    g = np.random.default_rng(6)
    prior = g.normal(size=(B, d, n))
    beng = _slope_engine(obe, prior, seed=seed)
    fa = _factor(g, d, zero_row=False)
    qa = fa @ fa.T
    qs = np.stack([qa * (b + 1) for b in range(B)])

    def update():
        x = _snapshot(beng)['p0'].reshape(d, B, beng._np)[:, :, :n]
        beng.pdf_update(np.zeros((B, 1)), sigma=1e12)          # flat: no resample, only the drift moves the cloud
        assert not beng.just_resampled.any()
        return x, _snapshot(beng)['p0'].reshape(d, B, beng._np)[:, :, :n]

    from optbayesexpt_b200.drift import drift_factor
    plan = [(qa, 1), (qs, 2), (None, 2), (qa, 3)]
    for drift, step in plan:
        beng.drift = drift
        x, y = update()
        assert beng._drift_step == step
        if drift is None:
            assert_array_equal(y, x)
            continue
        for b in range(B):
            f = drift_factor(drift if drift.ndim == 2 else drift[b], d)
            _check_moved(x[:, b], y[:, b], f, obd.batched_drift_normals(n, d, beng._seed_normal, step, b))


def test_c_entries_refuse_bad_input(obe):
    import torch
    from optbayesexpt_b200 import _lib
    lib = _lib.load()
    g = np.random.default_rng(1)
    beng = _slope_engine(obe, g.normal(size=(4, 3, 3000)))
    f = _lib.darr(np.eye(3).reshape(-1))
    fdev = torch.zeros((4, 3, 3), dtype=torch.float64, device='cuda')
    ok = dict(fh=f, fd=None, le=0, lt=0, ni=None, nn=0)

    def call(bs=None, **kw):
        a = dict(ok, **kw)
        return lib.obe_batch_drift(beng._bs() if bs is None else bs, a['fh'], a['fd'], a['le'], a['lt'], a['ni'],
                                   a['nn'], 1, 1, beng._stream())

    assert call() == 0
    assert call(fh=None, fd=C.c_void_p(fdev.data_ptr())) == 0
    cases = [
        (dict(bs=C.cast(None, _lib._PBATCH)), 'null'),
        (dict(fh=None), 'exactly one'),
        (dict(fd=C.c_void_p(fdev.data_ptr())), 'exactly one'),
        (dict(fh=_lib.darr(np.ones((3, 3)).reshape(-1))), 'lower-triangular'),
        (dict(fh=_lib.darr([np.nan] + [0.0] * 8)), 'finite'),
        (dict(ni=_lib.iarr([0]), nn=5), 'n_noise'),
        (dict(nn=1), 'n_noise'),
        (dict(ni=_lib.iarr([3]), nn=1), 'noise_index'),
    ]
    for kw, msg in cases:
        assert call(**kw) != 0, msg
        assert msg.encode() in lib.obe_last_error(), (msg, lib.obe_last_error())
    for field, value in (('d', 9), ('tiles', 3), ('n', 0), ('particles_dev', (C.c_void_p * 2)(None, None))):
        bad = _lib.Batch.from_buffer_copy(beng._batch)
        setattr(bad, field, value)
        assert call(bs=C.byref(bad)) != 0, field
    truth = torch.zeros((3, 4), dtype=torch.float64, device='cuda')
    tp = C.c_void_p(truth.data_ptr())
    s = beng._stream()
    assert lib.obe_batch_truth_drift(tp, 4, 4, 3, f, None, 1, 1, s) == 0
    for args, msg in (((None, 4, 4, 3, f, None), 'null truth'), ((tp, 3, 4, 3, f, None), 'ld_true'),
                      ((tp, 4, 4, 9, f, None), 'n_params'), ((tp, 4, 0, 3, f, None), 'n_inst'),
                      ((tp, 4, 4, 3, None, None), 'exactly one'),
                      ((tp, 4, 4, 3, _lib.darr(np.ones(9)), None), 'lower-triangular')):
        assert lib.obe_batch_truth_drift(*args, 1, 1, s) != 0, msg
        assert msg.encode() in lib.obe_last_error(), (msg, lib.obe_last_error())
    torch.cuda.synchronize()
    # the accepted call moved the zero truths by one step of the identity factor
    assert_allclose(_np(truth).T, obd.truth_walk(np.zeros((4, 3)), np.eye(3), 1, 1), rtol=1e-5, atol=1e-3)
