"""The device exp of the likelihood (obe_exp_nonpos_vec): <= 2 ulp against a correctly rounded exp over the whole
argument range the Gaussian log-likelihood can take, 0 below -708 and for NaN.

The update pass is driven through ``likelihood`` (obe_update_from_y with unit weights): with y_meas = 0 and sigma = 1
the exponent argument of particle i is exactly fl(-0.5 * y_i * y_i) and the stored weight is exactly its exp, so the
model rows y_i = sqrt(-2 x_i) sweep the argument over [-745, 0]."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def obe():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import optbayesexpt_b200 as pkg
    return pkg


def _exp_ref(x):
    """exp correctly rounded to float64 (through the 64-bit-mantissa long double), 0 where it is subnormal."""
    assert np.finfo(np.longdouble).nmant >= 63, 'the reference needs an extended-precision long double'
    ref = np.exp(x.astype(np.longdouble)).astype(np.float64)
    return np.where(ref < np.finfo(np.float64).tiny, 0.0, ref)


def _sweep():
    dense = np.linspace(-745.0, 0.0, 1 << 20)                       # every reduction interval ~23 times
    small = -np.geomspace(1e-300, 1.0, 1 << 16)                      # arguments near 0: r = x, k = 0
    cut = np.linspace(-708.5, -707.5, 1 << 12)                       # both sides of the underflow cut
    return np.concatenate([dense, small, cut, [0.0, -0.0, -708.0, -745.0, -1e4]])


def test_exp_within_2_ulp(obe):
    xs = _sweep()
    y = np.sqrt(-2.0 * xs)
    y_model = np.concatenate([y, [np.nan, np.inf]])
    n = y_model.size
    args = (-0.5 * y) * y                                            # what the kernel exponentiates, bit for bit
    g = np.random.default_rng(1)
    prior = np.array([g.uniform(2, 4, n), g.uniform(-2000, -400, n), g.normal(50000, 1000, n)])
    eng = obe.OptBayesExpt('lorentzian_hwhm', (np.linspace(1.5, 4.5, 16),), prior, (0.1,), scale=False,
                           default_noise_std=1.0, seed=3)
    got = eng.likelihood(y_model[None, :], (2.0, 0.0, 1.0))
    assert got.shape == (n,)
    # NaN and +inf model values (argument NaN and -inf) give an exact 0
    assert got[-2] == 0.0 and got[-1] == 0.0
    got = got[:-2]
    want = _exp_ref(args)
    below = args < -708.0
    assert np.all(got[below] == 0.0), 'arguments below -708 must give exactly 0'
    keep = ~below
    assert np.all(want[keep] > 0.0)
    ulp = np.abs(got[keep].view(np.int64) - want[keep].view(np.int64))
    worst = int(np.argmax(ulp))
    assert ulp.max() <= 2, f'{ulp.max()} ulp at x = {args[keep][worst]!r}: {got[keep][worst]!r} vs {want[keep][worst]!r}'
