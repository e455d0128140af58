"""CPU tests of the batch-statistics definitions: the numpy reference (oracle/stats_oracle.py) on
hand-made arrays, and the limit rows and accessors of BatchStats."""
import numpy as np
import pytest

import stats_oracle as S


def _one_row(x, status=None, q=(), limits=None):
    """Statistics of one V_m row: H = 1, n = 1, THD rows set to zero."""
    x = np.asarray(x, np.float64)
    B = x.size
    counts, st = S.batch_stats(x.reshape(1, 1, B), np.zeros((2, 1, B)), status, q,
                               None if limits is None else [limits, np.inf, np.inf])
    return counts, st[:, 0]


def _bits(v):
    return np.asarray(v, np.float64).view(np.uint64)


def test_order_keys_rank_negatives_zeros_and_ties():
    x = np.array([3.0, -1.0, 0.0, -0.0, -np.inf, 2.5, np.inf, -1.0])
    k = S.order_keys(x)
    order = np.argsort(k, kind="stable")
    assert list(_bits(x[order])) == list(_bits([-np.inf, -1.0, -1.0, -0.0, 0.0, 2.5, 3.0, np.inf]))
    assert S.order_keys(np.array([-0.0]))[0] + np.uint64(1) == S.order_keys(np.array([0.0]))[0]


def test_nearest_rank_quantiles_with_ties():
    x = [5.0, 1.0, 3.0, 3.0, 3.0, 2.0, 4.0, 3.0]             # sorted: 1 2 3 3 3 3 4 5
    q = (0.0, 0.1, 0.125, 0.126, 0.25, 0.5, 0.75, 0.76, 0.875, 0.9, 1.0)
    _, st = _one_row(x, q=q)
    want = [1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5]                  # value of rank max(1, ceil(p * 8))
    assert list(st[5:]) == want
    srt = np.sort(np.asarray(x))
    for p, v in zip(q, st[5:]):
        assert v == np.quantile(srt, p, method="inverted_cdf")
    assert st[2] == 1.0 and st[3] == 5.0


def test_signed_zeros_and_negatives():
    x = [0.0, -0.0, -2.0, 0.0, -0.0, -7.5]                    # key order: -7.5 -2 -0 -0 +0 +0
    _, st = _one_row(x, q=(0.0, 0.5, 0.51, 0.67, 1.0))          # ranks 1, 3, 4, 5, 6
    assert list(_bits(st[[2, 3]])) == list(_bits([-7.5, 0.0]))
    assert list(_bits(st[5:])) == list(_bits([-7.5, -0.0, -0.0, 0.0, 0.0]))
    _, st = _one_row([-0.0, 0.0], q=(0.5,))
    assert _bits(st[2]) == _bits(-0.0) and _bits(st[3]) == _bits(0.0) and _bits(st[5]) == _bits(-0.0)
    _, st = _one_row(x)
    assert st[0] == np.sum(x) / 6


def test_mean_std_exceed_and_masking():
    x = np.array([1.0, 2.0, 4.0, 100.0, 7.0])
    status = np.array([0, 0, 0, 1, 0])                         # the 100 is not converged
    counts, st = _one_row(x, status=status, q=(0.5,), limits=3.0)
    assert list(counts) == [4, 1, 0, 0]
    inc = x[status == 0]
    assert st[0] == inc.sum() / 4
    assert st[1] == np.sqrt(((inc - inc.mean()) ** 2).sum() / 4) == np.std(inc)
    assert st[2] == 1.0 and st[3] == 7.0 and st[4] == 2.0 and st[5] == 2.0
    counts, _ = _one_row(x, status=np.array([0, 3, 2, 1, 9]))
    assert list(counts) == [1, 1, 1, 1]                        # a value outside HPF_ST_* is not counted
    # +inf limit or no limit: never exceeded
    assert _one_row(x, limits=np.inf)[1][4] == 0.0 and _one_row(x)[1][4] == 0.0


@pytest.mark.parametrize("v", [1.0, 0.75, -3.5])
def test_constant_row_has_zero_std(v):
    """A constant row whose sum is exact (the slack bus's V_m = 1 is one): mean is the value, std exactly 0.
    (For other values the two-pass std of a constant row is the rounding error of the mean.)"""
    x = np.full(37, v)
    _, st = _one_row(x, q=(0.0, 0.3, 1.0))
    assert st[1] == 0.0 and st[0] == v and st[2] == st[3] == v
    assert (st[5:] == v).all()


def test_one_and_zero_included_scenarios():
    counts, st = _one_row([4.5, 9.0], status=np.array([2, 0]), q=(0.0, 0.5, 1.0), limits=5.0)
    assert list(counts) == [1, 0, 1, 0]
    assert st[0] == 9.0 and st[1] == 0.0 and st[2] == st[3] == 9.0 and st[4] == 1.0
    assert (st[5:] == 9.0).all()
    counts, st = _one_row([4.5, 9.0], status=np.array([1, 3]), q=(0.5,), limits=1.0)
    assert list(counts) == [0, 1, 0, 1]
    assert np.isnan(st[[0, 1, 2, 3, 5]]).all() and st[4] == 0.0
    counts, st = S.batch_stats(np.zeros((2, 3, 0)), np.zeros((2, 3, 0)), None, (0.5,))
    assert list(counts) == [0, 0, 0, 0] and st.shape == (6, 12)
    assert np.isnan(st[[0, 1, 2, 3, 5]]).all() and (st[4] == 0).all()


def test_row_layout_and_limit_rows():
    """Rows are V_m (h*n + i), THD_F, THD_R; BatchStats and stats_limit_rows use the same layout."""
    from harmonic_power_flow_b200.solver import BatchStats, stats_limit_rows
    H, n, B = 3, 2, 5
    rng = np.random.default_rng(0)
    V_m, thd = rng.uniform(0, 1, (H, n, B)), rng.uniform(0, 1, (2, n, B))
    lim = stats_limit_rows({"V_m": np.array([[0.5], [0.4], [0.3]]), "THD_F": 0.2}, n, H)
    assert lim.shape == (H * n + 2 * n,)
    assert list(lim[:H * n]) == [0.5, 0.5, 0.4, 0.4, 0.3, 0.3] and list(lim[H * n:]) == [0.2, 0.2, np.inf, np.inf]
    assert stats_limit_rows(None, n, H) is None
    with pytest.raises(ValueError):
        stats_limit_rows({"V_a": 1.0}, n, H)
    counts, st = S.batch_stats(V_m, thd, None, (0.5, 0.95), lim)
    bs = BatchStats(counts, (0.5, 0.95), st, n, H)
    assert np.array_equal(bs.V_m("max"), V_m.max(axis=2))
    assert np.array_equal(bs.THD_F("min"), thd[0].min(axis=1)) and np.array_equal(bs.THD_R("min"), thd[1].min(axis=1))
    assert np.array_equal(bs.V_m("exceed"), (V_m > lim[:H * n].reshape(H, n)[:, :, None]).sum(axis=2))
    assert np.array_equal(bs.THD_F(0.95), np.quantile(thd[0], 0.95, axis=1, method="inverted_cdf"))
