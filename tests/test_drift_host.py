"""CPU tests of the random-walk drift: argument validation, the factor F with F F^T = Q, the refusals of the sweeper and
the sharded engine, and the oracle's restatement of the drift normals' keying."""
import numpy as np
import pytest
from numpy.testing import assert_array_equal

from optbayesexpt_b200.drift import drift_factor, semidefinite_cholesky
from oracle import drift as odr
from oracle import obe_oracle as orc


@pytest.mark.parametrize('bad', [
    np.ones(2),                       # wrong number of standard deviations
    np.eye(2),                        # wrong covariance shape
    np.ones((3, 2)),
    np.ones((3, 3, 1)),
    [0.1, -0.2, 0.3],                 # negative standard deviation
    -1.0,
    [0.1, np.nan, 0.3],
    np.inf,
    [[1.0, 0.5, 0.0], [0.4, 1.0, 0.0], [0.0, 0.0, 1.0]],      # not symmetric
    [[1.0, 2.0, 0.0], [2.0, 1.0, 0.0], [0.0, 0.0, 1.0]],      # indefinite
    [[1.0, 0.0, 0.0], [0.0, -1e-3, 0.0], [0.0, 0.0, 1.0]],    # negative variance
    [[1.0, 0.0, np.nan], [0.0, 1.0, 0.0], [np.nan, 0.0, 1.0]],
    'abc',
])
def test_bad_drift_is_refused(bad):
    with pytest.raises(ValueError):
        drift_factor(bad, 3)


def test_none_is_no_drift():
    assert drift_factor(None, 3) is None


def test_standard_deviations_give_a_diagonal_factor():
    assert_array_equal(drift_factor(0.25, 3), np.diag([0.25, 0.25, 0.25]))
    assert_array_equal(drift_factor([0.1, 0.0, 2.0], 3), np.diag([0.1, 0.0, 2.0]))
    assert_array_equal(drift_factor([0.5], 1), [[0.5]])
    assert_array_equal(drift_factor([[0.25]], 1), [[0.5]])          # a (1, 1) array is a variance


def _check_factor(q, f):
    assert np.all(np.triu(f, 1) == 0.0), 'F must be lower-triangular'
    scale = np.max(np.abs(q))
    assert np.max(np.abs(f @ f.T - q)) <= 1e-12 * scale


@pytest.mark.parametrize('d', [1, 2, 3, 5, 8])
def test_factor_of_a_covariance(d):
    g = np.random.default_rng(d)
    for _ in range(20):
        a = g.normal(size=(d, d)) * np.exp(g.uniform(-3, 3, size=d))[:, None]
        q = a @ a.T
        f = drift_factor(q, d)
        _check_factor(q, f)
        assert np.all(np.diag(f) > 0.0)


def test_semidefinite_covariance_is_accepted():
    g = np.random.default_rng(7)
    for d, rank in [(2, 1), (3, 1), (3, 2), (5, 3), (8, 4)]:
        a = g.normal(size=(d, rank))
        q = a @ a.T
        _check_factor(q, drift_factor(q, d))
    _check_factor(np.ones((3, 3)), drift_factor(np.ones((3, 3)), 3))        # perfectly correlated steps
    assert_array_equal(drift_factor(np.zeros((2, 2)), 2), np.zeros((2, 2)))


def test_zero_variance_parameters_get_exactly_zero_rows():
    g = np.random.default_rng(3)
    a = g.normal(size=(5, 5))
    q = a @ a.T
    keep = [0, 2, 4]
    q[1, :] = q[:, 1] = 0.0
    q[3, :] = q[:, 3] = 0.0
    f = drift_factor(q, 5)
    _check_factor(q, f)
    assert np.all(f[1] == 0.0) and np.all(f[3] == 0.0)
    assert np.all(np.diag(f)[keep] > 0.0)
    assert np.all(drift_factor([0.3, 0.0, 0.1], 3)[1] == 0.0)
    # a rounding-level pivot counts as zero rather than producing a huge column
    low = semidefinite_cholesky([[1.0, 1.0], [1.0, 1.0 + 1e-17]])
    assert low[1, 1] == 0.0


def test_sweeper_and_sharded_refuse_drift():
    import optbayesexpt_b200 as obe
    from optbayesexpt_b200.sharded import ShardedOptBayesExpt
    prior = np.ones((3, 16))
    with pytest.raises(ValueError, match='drift'):
        obe.OptBayesExptSweeper('lorentzian_hwhm', (np.linspace(0, 1, 8),), prior, (1.0,), 2, drift=0.1)
    with pytest.raises(ValueError, match='drift'):
        ShardedOptBayesExpt('lorentzian_hwhm', (np.linspace(0, 1, 8),), prior, (1.0,), drift=[0.1, 0.0, 0.0])


def test_drift_normals_keying():
    n, d, seed, epoch = 200_000, 3, 12345, 7
    z = odr.drift_normals(n, d, seed, epoch)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01
    assert abs(np.corrcoef(z.T)[0, 1]) < 0.01
    # per-slot stream: any window of slots is the same numbers
    for dd in (1, 3, 5, 8):
        whole = odr.drift_normals(1000, dd, 99, 4)
        assert_array_equal(whole[337:911], odr.drift_normals(911 - 337, dd, 99, 4, slot_begin=337))
        assert_array_equal(whole[:, :min(dd, 4)], odr.drift_normals(1000, min(dd, 4), 99, 4))
    # every drift step draws new numbers, and none of them are the Liu-West jitter of the same seed and epoch
    assert not np.array_equal(odr.drift_normals(64, 3, 99, 4), odr.drift_normals(64, 3, 99, 5))
    assert not np.array_equal(odr.drift_normals(64, 3, 99, 4), odr.drift_normals(64, 3, 100, 4))
    ours = odr.drift_normals(4096, 3, 99, 4)
    for other in (orc.device_normals(4096, 3, 99, 4), orc.device_normals_packed(4096, 3, 99, 4)):
        assert np.abs(np.corrcoef(ours.reshape(-1), other.reshape(-1))[0, 1]) < 0.05
        assert not np.any(ours == other)
    # the counter word and the key both differ from the Liu-West stream's
    x = orc.philox4x32_10(np.uint32(5), np.uint32(0), np.uint32(odr.DRIFT_CTR), np.uint32(4),
                          (99 ^ odr.DRIFT_KEY) & 0xFFFFFFFF, (99 ^ odr.DRIFT_KEY) >> 32)
    y = orc.philox4x32_10(np.uint32(5), np.uint32(0), np.uint32(0), np.uint32(4), 99, 0)
    assert not np.array_equal(np.array(x), np.array(y))


def test_drift_step_restatement():
    x = np.array([[1.0, 0.1, -2.0], [3.0, 3.0, 3.0]])
    f = np.array([[0.5, 0.0], [0.2, 0.0]])
    z = np.array([[1.0, 9.0], [-1.0, 9.0], [2.0, 9.0]])
    moved, ok = odr.drift_step(x, f, z, mask_le=1)
    assert_array_equal(ok, [True, False, False])
    assert_array_equal(moved[:, 0], [1.5, 3.2])
    assert_array_equal(moved[:, 1:], x[:, 1:])
