"""numpy implementation of the correlated stochastic forcing contract (samsim_b200_set_stochastic_forcing_correlated,
samsim_b200/csrc/noise.cuh, DESIGN §7.4), written from the definition and independent of the C++ code.  The normals
are those of tests/stochastic_ref.py; det_log, det_cos and det_exp are passed in by the caller."""
import math

import numpy as np

import stochastic_ref as sref


def cholesky(corr):
    """L of the 4x4 corr by Cholesky-Banachiewicz, every operation a Python float (IEEE double, rounded on its own);
    None when a pivot is not > 0"""
    c = np.asarray(corr, dtype=np.float64).reshape(4, 4)
    L = [[0.0] * 4 for _ in range(4)]
    for i in range(4):
        for j in range(i + 1):
            s = float(c[i, j])
            for m in range(j):
                s = s - L[i][m] * L[j][m]
            if i == j:
                if not s > 0.0:
                    return None
                L[i][i] = math.sqrt(s)
            else:
                L[i][j] = s / L[j][j]
    return np.array(L)


def is_identity(corr):
    return corr is None or not (np.asarray(corr, dtype=np.float64).reshape(4, 4)[~np.eye(4, dtype=bool)] != 0.0).any()


def innovations(seed, corr, ids, nrec, det_log, det_cos):
    """w[k, b, r-1] of basis ids[b], records 1..nrec"""
    recs = np.arange(1, nrec + 1)
    z = np.stack([sref.normals(seed, k, ids, recs, det_log, det_cos) for k in range(4)])
    if is_identity(corr):
        return z
    L = cholesky(corr)
    w = np.empty_like(z)
    for k in range(4):
        s = L[k, 0] * z[0]
        for j in range(1, k + 1):
            s = s + L[k, j] * z[j]
        w[k] = s
    return w


def basis_series(seed, sigma, phi, corr, ids, nrec, det_log, det_cos):
    """E[k, b, r-1] of basis ids[b], records 1..nrec"""
    w = innovations(seed, corr, ids, nrec, det_log, det_cos)
    E = np.empty_like(w)
    for k in range(4):
        c = sigma[k] * np.sqrt(1.0 - phi[k] * phi[k])
        E[k, :, 0] = sigma[k] * w[k, :, 0]
        for r in range(1, nrec):
            E[k, :, r] = phi[k] * E[k, :, r - 1] + c * w[k, :, r]
    return E


def mix(basis, weights, ids, E):
    """the columns' e[c, r] from E[b, r] of one kind (rows in the order of ids), their q[c] and whether they have an
    entry; basis[c, m] ids or -1, weights[c, m]"""
    basis = np.asarray(basis).reshape(len(basis), -1)
    weights = np.ones(basis.shape) if weights is None else np.asarray(weights, dtype=np.float64).reshape(basis.shape)
    row = {int(b): j for j, b in enumerate(ids)}
    ncol, nmix = basis.shape
    e = np.zeros((ncol, E.shape[1]))
    q = np.zeros(ncol)
    has = np.zeros(ncol, dtype=bool)
    for c in range(ncol):
        for m in range(nmix):
            b = int(basis[c, m])
            if b < 0:
                continue
            w = weights[c, m]
            if has[c]:
                e[c] = e[c] + w * E[row[b]]
                q[c] = q[c] + w * w
            else:
                e[c] = w * E[row[b]]
                q[c] = w * w
            has[c] = True
    return e, q, has


def apply(mode, sigma, v, e, q, det_exp):
    """the record values v perturbed by a column's mixed e, q its sum of squared weights"""
    if mode == 0:
        return v + e
    if mode == 1:
        return v * np.fmax(1.0 + e, 0.0)
    x = np.asarray(e - (0.5 * (sigma * sigma)) * q, dtype=np.float64)
    return v * det_exp(x.ravel()).reshape(x.shape)


def noise(seed, sigma, phi, corr, basis, weights, nrec, det_log, det_cos):
    """e[k, c, r-1]: what samsim_b200_get_forcing_noise returns (0 for a column with no entry and for sigma 0)"""
    basis = np.asarray(basis).reshape(len(basis), -1)
    ids = np.unique(basis[basis >= 0])
    E = basis_series(seed, sigma, phi, corr, ids, nrec, det_log, det_cos)
    out = np.zeros((4, len(basis), nrec))
    for k in range(4):
        if sigma[k] != 0.0:
            out[k] = mix(basis, weights, ids, E[k])[0]
    return out


def perturbed(seed, sigma, phi, mode, corr, basis, weights, values, det_log, det_cos, det_exp):
    """values[c, 4, nrec] (base * scale + offset of column c) -> what column c reads, record by record"""
    out = np.array(values, dtype=np.float64, copy=True)
    basis = np.asarray(basis).reshape(len(basis), -1)
    ids = np.unique(basis[basis >= 0])
    E = basis_series(seed, sigma, phi, corr, ids, out.shape[2], det_log, det_cos)
    for k in range(4):
        if sigma[k] == 0.0:
            continue
        e, q, has = mix(basis, weights, ids, E[k])
        out[has, k] = apply(mode[k], sigma[k], out[has, k], e[has], q[has, None], det_exp)
    return out
