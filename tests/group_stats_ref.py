"""numpy implementation of the group statistics contract of include/samsim_b200.h (samsim_b200_set_group_stats):
the reference the GPU and host-compiled tests compare with, bit for bit."""
import numpy as np

from samsim_b200 import api

NSC = len(api.SNAP_SCALARS)


def tree(a):
    """pairwise sum along axis 0: pad with +0.0 to a power of two, then a = a[0::2] + a[1::2] repeated"""
    a = np.asarray(a, dtype=np.float64)
    n = a.shape[0]
    p = 1 if n <= 1 else 1 << (n - 1).bit_length()
    a = np.concatenate([a, np.zeros((p - n,) + a.shape[1:])])
    while a.shape[0] > 1:
        a = a[0::2] + a[1::2]
    return a[0]


def quantities(snap, depths, profiles):
    """values X[ncol, Q] of a snapshot and whether each lies above the member's ice bottom"""
    sc = np.stack([snap[n] for n in api.SNAP_SCALARS], 1)
    ncol = sc.shape[0]
    X = [sc]
    reached = [np.ones((ncol, NSC), dtype=bool)]
    if profiles:
        na = snap["N_active"].astype(int)
        kk = np.empty((ncol, len(depths)), dtype=int)
        for c in range(ncol):
            D = np.cumsum(snap["thick"][c, :na[c]])     # sequential, left to right
            kk[c] = np.searchsorted(D, depths, side="left")
        ok = kk < na[:, None]
        kc = np.minimum(kk, snap["thick"].shape[1] - 1)
        for p in profiles:
            X.append(np.take_along_axis(snap[p], kc, 1))
            reached.append(ok)
    return np.concatenate(X, 1), np.concatenate(reached, 1)


def reference_record(snap, status, end, i_rec, goc, ngroup, depths=(), profiles=()):
    X, R = quantities(snap, np.asarray(depths), profiles)
    return group_stats(X, R & ((status == 0) & (end >= i_rec))[:, None], goc, ngroup)


def group_stats(X, C, goc, ngroup):
    """[ngroup, Q, 5] = count, mean, variance, min, max of values X[ncol, Q] where C[ncol, Q] (contributes)"""
    Q = X.shape[1]
    out = np.empty((ngroup, Q, 5))
    for g in range(ngroup):
        m = np.flatnonzero(goc == g)
        x, c = X[m], C[m]
        n = c.sum(0).astype(np.float64)
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = tree(np.where(c, x, 0.0)) / n
            d = np.where(c, x - mean, 0.0)
            m2 = tree(d * d)
            var = np.where(n >= 2, m2 / (n - 1), np.where(n == 1, 0.0, np.nan))
        mean = np.where(n > 0, mean, np.nan)
        xm = np.where(c, x, np.nan)
        mn = np.fmin.reduce(xm, axis=0) if len(m) else np.full(Q, np.nan)
        mx = np.fmax.reduce(xm, axis=0) if len(m) else np.full(Q, np.nan)
        out[g] = np.stack([n, mean, var, mn, mx], 1)
    return out
