"""CPU tests of the posterior summaries: the numpy oracle (oracle/summaries.py) against numpy's own weighted
quantile and histograms, its edge cases, and the argument checks of the Python layer."""
import numpy as np
import pytest

from oracle import summaries as orc


def _cloud(n, seed):
    g = np.random.default_rng(seed)
    x = g.normal(0.0, 1.0, n)
    w = g.exponential(size=n) ** 2
    return x, w / w.sum()


@pytest.mark.parametrize('n,seed', [(1, 0), (7, 1), (1000, 2), (100_003, 3)])
def test_quantile_oracle_against_numpy_inverted_cdf(n, seed):
    x, w = _cloud(n, seed)
    levels = np.concatenate([[0.0, 0.025, 0.5, 0.975, 1.0], np.random.default_rng(seed).random(11)])
    got = orc.quantile(x, orc.quantised(w), levels)
    want = np.quantile(x, levels, weights=w, method='inverted_cdf')
    differ = got != want
    if np.any(differ):
        # only where the float cumulative weight sits within 1e-10 of q at the crossing
        order = np.argsort(x, kind='stable')
        cdf = np.cumsum(w[order]) / np.sum(w)
        for q in levels[differ]:
            i = np.searchsorted(cdf, q, side='left')
            near = [abs(cdf[k] - q) for k in (i - 1, i) if 0 <= k < n]
            assert min(near) <= 1e-10, f'q={q}: oracle {got[levels == q]} numpy {want[levels == q]}'


def test_quantile_definition_edges():
    x = np.array([3.0, -1.0, 2.0, 2.0, 5.0, -4.0])
    w = np.array([0.0, 0.25, 0.25, 0.25, 0.25, 0.0])             # zero-weight particles at both extremes
    wq = orc.quantised(w)
    np.testing.assert_array_equal(orc.quantile(x, wq, [0.0, 1.0]), [-1.0, 5.0])
    np.testing.assert_array_equal(orc.quantile(x, wq, [0.25, 0.2500001, 0.5, 0.75, 0.75000001]),
                                  [-1.0, 2.0, 2.0, 2.0, 5.0])
    same = np.full(10, 7.5)
    np.testing.assert_array_equal(orc.quantile(same, orc.quantised(np.full(10, 0.1)), [0, 0.3, 1]), [7.5] * 3)
    zeros = np.array([-0.0, 0.0, -0.0])
    r = orc.quantile(zeros, orc.quantised(np.full(3, 1 / 3)), [0.0, 0.5, 1.0])
    assert np.all(r == 0.0) and not np.any(np.signbit(r))
    with pytest.raises(ValueError):
        orc.quantile(x, np.zeros(6, dtype=np.uint64), [0.5])


def test_target_is_exact():
    W = 2 ** 62 + 12345
    assert orc.target(0.0, W) == 1
    assert orc.target(1.0, W) == W
    assert orc.target(0.5, W) == (W + 1) // 2
    assert orc.target(1e-300, W) == 1
    q = 0.1
    from fractions import Fraction
    assert orc.target(q, W) == -(-Fraction(q).numerator * W // Fraction(q).denominator)


def test_oversized_weight_total_is_refused():
    wq = orc.quantised(np.ones(8))                               # un-normalised: W = 8 * 2^62 wraps to 0 in 64 bits
    with pytest.raises(ValueError, match='sum to 4'):
        orc.quantile(np.arange(8.0), wq, [0.5])
    assert orc.total(orc.quantised(np.full(4, 0.99))) < 2 ** 64


def test_quantised_rounding():
    w = np.array([0.0, -1e-3, 2.0 ** -63, 3 * 2.0 ** -63, 1e-20, 0.25, 1.0])
    np.testing.assert_array_equal(orc.quantised(w), np.array([0, 0, 0, 2, 0, 2 ** 60, 2 ** 62], dtype=np.uint64))


@pytest.mark.parametrize('bins', [1, 7, 256, 4096])
def test_histogram_oracle_against_numpy(bins):
    x, w = _cloud(200_001, bins)
    x[:10] = x.min()                                             # values on the first and the last edge
    x[10:20] = x.max()
    wq = orc.quantised(w)
    e = np.histogram_bin_edges(x, bins)
    raw, cnt = orc.histogram(x, wq, e)
    # integer bins: numpy's uniform-bin path (an edge array would take its cumulative-sum path)
    np.testing.assert_array_equal(cnt, np.histogram(x, bins)[0])
    mass, ref = orc.mass(raw), np.histogram(x, bins, weights=w)[0]
    bound = 1e-12 * np.abs(ref) + cnt * 2.0 ** -63
    assert np.all(np.abs(mass - ref) <= bound)
    # explicit range narrower than the data: outside values dropped
    e2 = np.histogram_bin_edges(x, bins, range=(-0.5, 0.75))
    np.testing.assert_array_equal(orc.histogram(x, wq, e2)[1], np.histogram(x, bins, range=(-0.5, 0.75))[0])


def test_histogram2d_oracle_against_numpy():
    g = np.random.default_rng(5)
    x, y = g.normal(size=50_000), g.uniform(-1, 1, 50_000)
    w = g.random(50_000)
    w /= w.sum()
    x[:5] = 4.0                                                  # outside the range below
    H, xe, ye = np.histogram2d(x, y, bins=(33, 17), range=[[-3, 3], [-1, 1]], weights=w)
    C_, _, _ = np.histogram2d(x, y, bins=(33, 17), range=[[-3, 3], [-1, 1]])
    raw, cnt = orc.histogram2d(x, y, orc.quantised(w), xe, ye)
    np.testing.assert_array_equal(cnt, C_)
    assert np.all(np.abs(orc.mass(raw) - H) <= 1e-12 * H + cnt * 2.0 ** -63)
    from optbayesexpt_b200.summaries import edges_for
    np.testing.assert_array_equal(edges_for(-3, 3, 33), xe)


def test_u64_bincount_is_exact():
    g = np.random.default_rng(6)
    wq = g.integers(0, 2 ** 62, 100_000, dtype=np.uint64)
    idx = g.integers(-1, 5, 100_000)
    got, cnt = orc.u64_bincount(idx, wq, 5)
    for b in range(5):
        assert int(got[b]) == sum(int(v) for v in wq[idx == b]) % 2 ** 64
        assert cnt[b] == np.count_nonzero(idx == b)


def test_python_argument_checks():
    from optbayesexpt_b200 import summaries as s
    np.testing.assert_array_equal(s.quantile_levels(0.5), [0.5])
    assert s.quantile_levels([0, 1]).shape == (2,)
    for bad in ([], np.zeros(17), [1.5], [-0.1], [np.nan], [[0.5]]):
        with pytest.raises(ValueError):
            s.quantile_levels(bad)
    assert s.param_list(None, 3) == [0, 1, 2]
    assert s.param_list(2, 3) == [2]
    assert s.param_list([1, 0], 3) == [1, 0]
    for bad in ([3], [-1], 5, list(range(9))):
        with pytest.raises(ValueError):
            s.param_list(bad, 3 if bad != list(range(9)) else 8)
    for bad in (True, 1.5, 'x'):
        with pytest.raises(TypeError):
            s.param_list(bad, 3)
    assert s.hist_bins(4096) == 4096
    for bad in (0, 4097, -3):
        with pytest.raises(ValueError):
            s.hist_bins(bad)
    with pytest.raises(TypeError):
        s.hist_bins('auto')
    assert s.hist_bins2d(128) == (128, 128)
    assert s.hist_bins2d((16, 4096)) == (16, 4096)
    with pytest.raises(ValueError):
        s.hist_bins2d((257, 256))
    with pytest.raises(TypeError):
        s.hist_bins2d((1, 2, 3))
    assert s.hist_ranges(None, 2) is None
    assert s.hist_ranges((0, 1), 3) == [(0.0, 1.0)] * 3
    with pytest.raises(ValueError):
        s.hist_ranges([(0, 1)] * 2, 3)
    with pytest.raises(ValueError):
        s.edges_for(1.0, 0.0, 4)                                 # numpy's own range checks
    with pytest.raises(ValueError):
        s.edges_for(0.0, np.inf, 4)
    np.testing.assert_array_equal(s.edges_for(2.0, 2.0, 2), [1.5, 2.0, 2.5])


def test_sharded_engines_refuse_summaries():
    from optbayesexpt_b200.sharded import ShardedOptBayesExpt
    for call in (lambda: ShardedOptBayesExpt.quantile(None, 0.5), lambda: ShardedOptBayesExpt.histogram(None, 8),
                 lambda: ShardedOptBayesExpt.histogram2d(None, 0, 1, 8)):
        with pytest.raises(NotImplementedError, match='all-reduce'):
            call()


def test_batched_engines_have_no_summaries():
    from optbayesexpt_b200.batched import BatchedOptBayesExpt
    assert not any(hasattr(BatchedOptBayesExpt, m) for m in ('quantile', 'histogram', 'histogram2d'))
