"""CPU tests of the batched engines' random-walk drift: argument validation in the constructor and in set_simulator
(before any device is touched), the per-instance factors, and the oracle's restatement of the batched keying and of
the simulator's truth walk."""
import numpy as np
import pytest
from numpy.testing import assert_array_equal

from optbayesexpt_b200.drift import batched_drift_factors, drift_factor
from oracle import batched_drift as obd
from oracle import drift as odr
from oracle import obe_oracle as orc

B, D = 4, 3


def _spd(g, d):
    a = g.normal(size=(d, d))
    return a @ a.T


def _per_instance(bad_b, bad_q):
    g = np.random.default_rng(1)
    qs = np.stack([_spd(g, D) for _ in range(B)])
    qs[bad_b] = bad_q
    return qs


BAD = [
    np.ones(2),                                       # wrong number of standard deviations
    np.eye(2),                                        # wrong covariance shape
    np.ones((3, 2)),
    np.ones((B, D, D, 1)),
    np.ones((B + 1, D, D)),                           # per-instance: wrong number of instances
    np.ones((B, D - 1, D - 1)),
    np.ones((B, D)),                                  # per-instance standard deviations go as diagonal covariances
    [0.1, -0.2, 0.3],                                 # negative standard deviation
    -1.0,
    [0.1, np.nan, 0.3],
    np.inf,
    [[1.0, 0.5, 0.0], [0.4, 1.0, 0.0], [0.0, 0.0, 1.0]],      # not symmetric
    [[1.0, 2.0, 0.0], [2.0, 1.0, 0.0], [0.0, 0.0, 1.0]],      # indefinite
    'abc',
    _per_instance(2, np.nan),
    _per_instance(1, [[1.0, 0.5, 0.0], [0.4, 1.0, 0.0], [0.0, 0.0, 1.0]]),
    _per_instance(3, [[1.0, 2.0, 0.0], [2.0, 1.0, 0.0], [0.0, 0.0, 1.0]]),
    _per_instance(0, np.diag([1.0, -1e-3, 1.0])),
]


@pytest.mark.parametrize('bad', BAD)
def test_bad_drift_is_refused_by_the_constructor(bad):
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    prior = np.ones((B, D, 64))
    with pytest.raises(ValueError):
        BatchedOptBayesExpt('lorentzian_hwhm', (np.linspace(0, 1, 8),), prior, (1.0,), drift=bad)


@pytest.mark.parametrize('bad', BAD)
def test_bad_drift_is_refused_by_set_simulator(bad):
    import torch
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    from optbayesexpt_b200.models import builtin
    # an engine object without its device state: set_simulator must refuse before it needs any
    beng = object.__new__(BatchedOptBayesExpt)
    beng._torch = torch
    beng.n_instances = B
    beng.model_function = builtin('lorentzian_hwhm')         # n_model_params = 3 = D
    with pytest.raises(ValueError):
        beng.set_simulator(np.ones((B, D)), 1.0, drift=bad)


def test_none_is_no_drift():
    assert batched_drift_factors(None, B, D) is None


def test_shared_forms_give_the_single_engine_factor():
    q = _spd(np.random.default_rng(2), D)
    for drift in (0.3, [0.1, 0.0, 0.2], q, q.tolist()):
        assert_array_equal(batched_drift_factors(drift, B, D), drift_factor(drift, D))
    # n_instances == n_dims: a 2-D array is one shared covariance, never per-instance standard deviations
    assert_array_equal(batched_drift_factors(q, D, D), drift_factor(q, D))


def test_per_instance_factors_are_those_of_each_slice():
    g = np.random.default_rng(3)
    qs = np.stack([_spd(g, D) for _ in range(B)])
    qs[1] = np.diag([0.04, 0.0, 0.01])                # per-instance standard deviations as a diagonal covariance
    qs[2] = 0.0                                       # an instance that does not drift
    qs[3][1, :] = qs[3][:, 1] = 0.0                   # one parameter of one instance that does not drift
    f = batched_drift_factors(qs, B, D)
    assert f.shape == (B, D, D)
    for b in range(B):
        assert_array_equal(f[b], drift_factor(qs[b], D))
    assert_array_equal(f[1], np.diag([0.2, 0.0, 0.1]))
    assert_array_equal(f[2], 0.0)
    assert np.all(f[3][1] == 0.0)


def test_batched_keying():
    n, d, seed, step = 5000, 3, 0x1234567890ABCDEF, 9
    z = {b: obd.batched_drift_normals(n, d, seed, step, b) for b in range(4)}
    # instance b is slot (b << 32) | i of the single engine's keying
    assert_array_equal(z[2], odr.drift_normals(n, d, seed, step, slot_begin=2 << 32))
    assert_array_equal(z[0], odr.drift_normals(n, d, seed, step))
    allz = np.concatenate([z[b] for b in range(4)])
    assert abs(allz.mean()) < 0.02 and abs(allz.std() - 1.0) < 0.02
    # fresh numbers per instance, per step and per seed
    others = [obd.batched_drift_normals(n, d, seed, step + 1, 2), obd.batched_drift_normals(n, d, seed + 1, step, 2)]
    others += [z[b] for b in (0, 1, 3)]
    for other in others:
        assert not np.any(z[2] == other)
        assert abs(np.corrcoef(z[2].reshape(-1), other.reshape(-1))[0, 1]) < 0.05
    # the high slot word keeps every instance but 0 off the single engine's stream of slots 0 .. n-1
    single = odr.drift_normals(n, d, seed, step)
    for b in (1, 2, 3):
        assert not np.any(z[b] == single)


def test_truth_walk_keying():
    n_inst, npm, seed = 4096, 3, 12345
    t = obd.truth_normals(n_inst, npm, seed, 1)
    assert abs(t.mean()) < 0.03 and abs(t.std() - 1.0) < 0.03
    assert not np.any(t == obd.truth_normals(n_inst, npm, seed, 2))
    assert not np.any(t == obd.truth_normals(n_inst, npm, seed + 1, 1))
    # nothing in common with the particle drift, the Liu-West jitter or the simulator's measurement noise (all
    # drawn per instance / slot b with the same seed and step or cycle)
    for other in (odr.drift_normals(n_inst, npm, seed, 1), obd.batched_drift_normals(n_inst, npm, seed, 1, 0),
                  orc.device_normals(n_inst, npm, seed, 1)):
        assert not np.any(t == other)
        assert abs(np.corrcoef(t.reshape(-1), other.reshape(-1))[0, 1]) < 0.05
    x = orc.philox4x32_10(np.uint32(5), np.uint32(0), np.uint32(obd.TRUTH_CTR), np.uint32(1),
                          (seed ^ obd.TRUTH_KEY) & 0xFFFFFFFF, (seed ^ obd.TRUTH_KEY) >> 32)
    for word, key in ((odr.DRIFT_CTR, seed ^ odr.DRIFT_KEY), (0, seed)):
        y = orc.philox4x32_10(np.uint32(5), np.uint32(0), np.uint32(word), np.uint32(1), key & 0xFFFFFFFF, key >> 32)
        assert not np.array_equal(np.array(x), np.array(y))


def test_truth_walk_restatement():
    g = np.random.default_rng(4)
    x0 = g.normal(size=(6, 3))
    f = drift_factor(_spd(g, 3) * 0.01, 3)
    five = obd.truth_walk(x0, f, 7, 5)
    assert_array_equal(obd.truth_walk(obd.truth_walk(x0, f, 7, 2), f, 7, 3, first_step=3), five)
    assert_array_equal(obd.truth_walk(x0, f, 7, 0), x0)
    one = obd.truth_walk(x0, f, 7, 1)
    assert np.allclose(one, x0 + obd.truth_normals(6, 3, 7, 1) @ f.T, rtol=0, atol=1e-15)
    # per-instance factors: instance b walks with its own F
    fs = np.stack([f * (b + 1) for b in range(6)])
    per = obd.truth_walk(x0, fs, 7, 1)
    assert np.allclose(per - x0, (one - x0) * np.arange(1, 7)[:, None], rtol=1e-12, atol=1e-15)
