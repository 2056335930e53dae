"""numpy implementation of the time statistics contract of include/samsim_b200.h (samsim_b200_set_time_stats): the
reference the GPU and host-compiled tests compare with, bit for bit.  The Welford recurrence runs element by element in
float64, one record at a time; the regrid is that of the group statistics (group_stats_ref.quantities)."""
import numpy as np

from samsim_b200 import api
from group_stats_ref import NSC, quantities

STATS = ("count", "mean", "var", "min", "max")


def fmin(m, x):
    """fmin(m, x) with the tie of the contract: of two equal values (+0.0 and -0.0) m stays.  np.fmin itself picks
    either zero depending on its code path (scalar or array), so the rule is spelled out here."""
    return np.where((x < m) | np.isnan(m), x, m)


def fmax(m, x):
    return np.where((x > m) | np.isnan(m), x, m)


class Acc:
    """accumulators of the window in progress, any shape"""

    def __init__(self, shape):
        self.n, self.mean, self.m2 = np.zeros(shape), np.zeros(shape), np.zeros(shape)
        self.mn, self.mx = np.full(shape, np.nan), np.full(shape, np.nan)

    def update(self, x, c):
        """one record: values x where c (contributes)"""
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            n = self.n + 1.0
            d = x - self.mean
            mean = self.mean + d / n
            m2 = self.m2 + d * (x - mean)
        self.n, self.mean, self.m2 = np.where(c, n, self.n), np.where(c, mean, self.mean), np.where(c, m2, self.m2)
        self.mn, self.mx = np.where(c, fmin(self.mn, x), self.mn), np.where(c, fmax(self.mx, x), self.mx)

    def finish(self):
        """[..., 5] = count, mean, variance, min, max"""
        n = self.n
        with np.errstate(invalid="ignore", divide="ignore"):
            var = np.where(n >= 2, self.m2 / (n - 1), np.where(n == 1, 0.0, np.nan))
        mean = np.where(n > 0, self.mean, np.nan)
        return np.stack([n, mean, var, self.mn, self.mx], -1)


def record_values(snap, status, end, i_rec, scalars=None, depths=(), profiles=()):
    """values X[ncol, Q] of one record and whether each contributes: the selected scalars in id order, then the
    profiles on the depths; a column contributes when its status is 0 and its end step is >= i_rec"""
    X, R = quantities(snap, np.asarray(depths, dtype=np.float64), list(profiles))
    names = api.SNAP_SCALARS if scalars is None else scalars
    cols = sorted(api.SNAP_SCALARS.index(n) for n in names) + list(range(NSC, X.shape[1]))
    live = (np.asarray(status) == 0) & (np.asarray(end) >= i_rec)
    return X[:, cols], R[:, cols] & live[:, None]


def reference(records, windows, **sel):
    """records: [(i, snapshot, status, end steps)] in record order; windows: lists of record indices, each one window.
    Returns [W, ncol, Q, 5]."""
    out = []
    for w in windows:
        acc = None
        for r in w:
            i, snap, status, end = records[r]
            X, C = record_values(snap, status, end, i, **sel)
            if acc is None:
                acc = Acc(X.shape)
            acc.update(X, C)
        out.append(acc.finish())
    return np.stack(out)
