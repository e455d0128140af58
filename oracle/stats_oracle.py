"""Numpy reference of the batch statistics (hpf_batch_stats / hpf_solve_host_stats), with exactly the
definitions of include/hpf_b200.h.  Test infrastructure: the product never routes through it."""
from __future__ import annotations

import numpy as np


def order_keys(x):
    """Order-preserving uint64 keys of doubles: sign bit set on non-negative values, every bit flipped
    on negative ones (-0 sorts below +0).  The total order the batch statistics rank values by."""
    u = np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)
    return np.where(u >> np.uint64(63), ~u, u | np.uint64(1 << 63))


def batch_stats(V_m, thd, status=None, quantiles=(), limits=None):
    """Statistics of a batch as hpf_batch_stats defines them.  V_m [H, n, B], thd [2, n, B] (THD as
    hpf_thd writes it: a numpy restatement differs in the last bit where nvcc contracts to an FMA),
    status [B] or None (all included), limits [R] or None.  Rows: V_m (h*n + i), THD_F, THD_R.
    -> (status_counts [4] int, stats [5 + K, R]): mean, population std (two passes), min, max, exceed
    (x > limit), then the value of rank max(1, ceil(p * n_valid)) for every level p (nearest rank,
    numpy's method="inverted_cdf"), ranked by order_keys.  No included scenario: NaN, exceed 0."""
    V_m, thd = np.asarray(V_m, np.float64), np.asarray(thd, np.float64)
    H, n, B = V_m.shape
    X = np.concatenate([V_m.reshape(H * n, B), thd.reshape(2 * n, B)])
    R = X.shape[0]
    if status is None:
        counts = np.array([B, 0, 0, 0], np.int64)
        inc = np.ones(B, bool)
    else:
        status = np.asarray(status)
        counts = np.array([(status == s).sum() for s in range(4)], np.int64)
        inc = status == 0
    q = np.asarray(quantiles, np.float64).ravel()
    lim = np.full(R, np.inf) if limits is None else np.asarray(limits, np.float64)
    x = X[:, inc]
    nv = x.shape[1]
    out = np.full((5 + q.size, R), np.nan)
    out[4] = 0.0
    if nv == 0:
        return counts, out
    mean = x.sum(axis=1) / nv
    out[0] = mean
    out[1] = np.sqrt(((x - mean[:, None]) ** 2).sum(axis=1) / nv)
    srt = np.take_along_axis(x, np.argsort(order_keys(x), axis=1, kind="stable"), axis=1)
    out[2], out[3] = srt[:, 0], srt[:, -1]
    out[4] = (x > lim[:, None]).sum(axis=1)
    for k, p in enumerate(q):
        out[5 + k] = srt[:, max(1, int(np.ceil(p * float(nv)))) - 1]
    return counts, out
