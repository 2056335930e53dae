"""numpy implementation of the stochastic forcing contract (samsim_b200/csrc/noise.cuh, include/samsim_b200.h),
written from the definition and independent of the C++ code.  det_log, det_cos and det_exp are the deterministic
functions of detmath.h, passed in by the caller (the host build of tests/hostbuild/noise_on_host.cpp)."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)
S32 = np.uint64(32)


def philox(ctr, key):
    """Philox4x32-10 of counters ctr[..., 4] and keys key[..., 2] (broadcast), uint32 words -> uint32[..., 4]"""
    c = [np.asarray(ctr, dtype=np.uint64)[..., j] for j in range(4)]
    k = [np.asarray(key, dtype=np.uint64)[..., j] for j in range(2)]
    for rnd in range(10):
        if rnd:
            k = [(k[0] + W0) & MASK, (k[1] + W1) & MASK]
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> S32) ^ c[1] ^ k[0], p1 & MASK, (p0 >> S32) ^ c[3] ^ k[1], p0 & MASK]
    return np.stack(np.broadcast_arrays(*c), -1).astype(np.uint32)


def uniform(a, b):
    a, b = np.asarray(a, dtype=np.uint32) >> 6, np.asarray(b, dtype=np.uint32) >> 6
    return (a.astype(np.float64) * 2.0 ** 26 + b.astype(np.float64) + 0.5) * 2.0 ** -52


def normals(seed, kind, streams, recs, det_log, det_cos):
    """z[s, r] for streams[s] and records recs[r]"""
    s = np.asarray(streams, dtype=np.uint64)[:, None]
    r = np.asarray(recs, dtype=np.uint64)[None, :]
    ctr = np.stack(np.broadcast_arrays(r, np.uint64(kind), s, np.uint64(0)), -1)
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64)
    x = philox(ctr, key)
    u1, u2 = uniform(x[..., 0], x[..., 1]), uniform(x[..., 2], x[..., 3])
    lg = det_log(u1.ravel()).reshape(u1.shape)
    cs = det_cos((6.283185307179586 * u2).ravel()).reshape(u2.shape)
    return np.sqrt(-2.0 * lg) * cs


def series(seed, sigma, phi, kind, streams, nrec, det_log, det_cos):
    """e[s, r-1] for records r = 1..nrec; streams < 0 give 0"""
    streams = np.asarray(streams)
    z = normals(seed, kind, np.maximum(streams, 0), np.arange(1, nrec + 1), det_log, det_cos)
    c = sigma * np.sqrt(1.0 - phi * phi)
    e = np.empty_like(z)
    e[:, 0] = sigma * z[:, 0]
    for r in range(1, nrec):
        e[:, r] = phi * e[:, r - 1] + c * z[:, r]
    e[streams < 0] = 0.0
    return e


def apply(mode, sigma, v, e, det_exp):
    """the record values v perturbed by e"""
    if mode == 0:
        return v + e
    if mode == 1:
        return v * np.fmax(1.0 + e, 0.0)
    h = 0.5 * (sigma * sigma)
    x = np.asarray(e - h, dtype=np.float64)
    return v * det_exp(x.ravel()).reshape(x.shape)


def perturbed(seed, sigma, phi, mode, streams, values, det_log, det_cos, det_exp):
    """values[c, 4, nrec] (base * scale + offset of column c) -> what column c reads, record by record"""
    out = np.array(values, dtype=np.float64, copy=True)
    streams = np.asarray(streams)
    on = streams >= 0
    for k in range(4):
        if sigma[k] == 0.0 or not on.any():
            continue
        e = series(seed, sigma[k], phi[k], k, streams[on], out.shape[2], det_log, det_cos)
        out[on, k] = apply(mode[k], sigma[k], out[on, k], e, det_exp)
    return out
