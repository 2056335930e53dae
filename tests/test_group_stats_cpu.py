"""Group statistics without a GPU: the rules of samsim_b200/csrc/group_stats.cuh compiled for the host against the numpy
reference (tests/group_stats_ref.py), and distributed.reduce_group_stats over gloo at world sizes 2 and 3."""
import ctypes as C
import os
import subprocess
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
sys.path.insert(0, str(HERE))
from group_stats_ref import group_stats, tree  # noqa: E402

SRC = HERE / "hostbuild" / "group_stats_on_host.cpp"
LIB = HERE / "hostbuild" / "_build" / "libgroup_stats_on_host.so"
TILE = 1024


@pytest.fixture(scope="module")
def lib():
    deps = [SRC, ROOT / "samsim_b200" / "csrc" / "group_stats.cuh"]
    if not (LIB.exists() and all(LIB.stat().st_mtime > d.stat().st_mtime for d in deps)):
        LIB.parent.mkdir(exist_ok=True)
        r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-o", str(LIB), str(SRC)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    L = C.CDLL(str(LIB))
    i32, i64, dp = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    L.gsh_layout.restype = C.c_int64
    L.gsh_layout.argtypes = [C.c_int64, C.c_int32, i32, i32, i32, C.c_int64, i64, i32]
    L.gsh_regrid.restype = C.c_double
    L.gsh_regrid.argtypes = [dp, C.c_int32, dp, C.c_int32, i32]
    L.gsh_finish.argtypes = [C.c_int32, dp, dp, dp, dp, dp]
    return L


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def layout(L, goc, ngroup):
    goc = np.ascontiguousarray(goc, dtype=np.int32)
    npad = L.gsh_layout(len(goc), ngroup, _p(goc, C.c_int32), None, None, 0, None, None)
    col, info = np.empty(npad, np.int32), np.empty(npad, np.int32)
    start, lg = np.empty(ngroup, np.int64), np.empty(ngroup, np.int32)
    L.gsh_layout(len(goc), ngroup, _p(goc, C.c_int32), _p(col, C.c_int32), _p(info, C.c_int32), npad,
                 _p(start, C.c_int64), _p(lg, C.c_int32))
    return col, info, start, lg


def tiled_sums(x, start, lg):
    """the sums the GPU forms on the padded layout: the tree inside each tile of TILE entries (a whole group or one
    aligned chunk of a larger group), then the tree over the chunk sums"""
    out = []
    for s, l in zip(start, lg):
        p = 1 << int(l)
        seg = x[s:s + p]
        if p <= TILE:
            out.append(tree(seg))
        else:
            out.append(tree(np.array([tree(seg[k:k + TILE]) for k in range(0, p, TILE)])))
    return np.array(out)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_layout_makes_the_tiled_tree_the_whole_tree(lib, seed):
    rng = np.random.default_rng(seed)
    sizes = [1, 0, 3000, 1024, 1025, 20, 17, 16, 0, 2, 5000, 33, 64, 1] + list(rng.integers(0, 40, 30))
    ngroup = len(sizes)
    goc = np.concatenate([np.full(n, g) for g, n in enumerate(sizes)] + [np.full(77, -1)]).astype(np.int32)
    rng.shuffle(goc)
    col, info, start, lg = layout(lib, goc, ngroup)
    assert len(col) % TILE == 0
    vals = rng.normal(size=len(goc)) * 10.0 ** rng.integers(-8, 8, len(goc))
    vals[rng.random(len(goc)) < 0.05] = -0.0
    for g, n in enumerate(sizes):
        p = 1 << int(lg[g])
        assert p == max(1, 1 << int(np.ceil(np.log2(max(n, 1)))))
        assert start[g] % p == 0
        members = np.flatnonzero(goc == g)
        assert np.array_equal(col[start[g]:start[g] + n], members)          # ascending caller column order
        assert (col[start[g] + n:start[g] + p] == -1).all()
        assert (info[start[g]:start[g] + p] == (g << 5 | lg[g])).all()
    used = np.zeros(len(col), bool)
    for g in range(ngroup):
        used[start[g]:start[g] + (1 << int(lg[g]))] = True
    assert (info[~used] == -1).all() and (col[~used] == -1).all()
    x = np.where(col >= 0, vals[np.maximum(col, 0)], 0.0)
    whole = np.array([tree(vals[goc == g]) if sizes[g] else 0.0 for g in range(ngroup)])
    assert np.array_equal(bits(tiled_sums(x, start, lg)), bits(whole))


def test_group_of_all_columns(lib):
    col, info, start, lg = layout(lib, np.zeros(70_000, np.int32), 1)
    assert lg[0] == 17 and start[0] == 0 and len(col) == 1 << 17
    assert np.array_equal(col[:70_000], np.arange(70_000))


def test_regrid_matches_numpy(lib):
    rng = np.random.default_rng(4)
    for trial in range(300):
        n = int(rng.integers(0, 40))
        thick = rng.uniform(0.0, 0.2, 45)
        thick[rng.random(45) < 0.1] = 0.0
        na = int(rng.integers(0, n + 1))
        D = np.cumsum(thick[:na])
        z = np.sort(np.unique(np.concatenate([rng.uniform(1e-3, 5.0, 12), D[D > 0][:3]])))   # some exactly on D_k
        layer = np.empty(len(z), np.int32)
        reach = lib.gsh_regrid(_p(np.ascontiguousarray(thick), C.c_double), na, _p(z, C.c_double), len(z),
                               _p(layer, C.c_int32))
        k = np.searchsorted(D, z, side="left")
        expect = np.where(k < na, k + 1, 0)
        assert np.array_equal(layer, expect), trial
        assert reach == (D[-1] if na else 0.0)


def test_finish_matches_numpy(lib):
    rng = np.random.default_rng(5)
    n = np.array([0, 1, 2, 3, 1000], dtype=np.float64)
    s, m2 = rng.normal(size=5), rng.uniform(0, 1, 5)
    mean, var = np.empty(5), np.empty(5)
    lib.gsh_finish(5, *[_p(a, C.c_double) for a in (n, s, m2, mean, var)])
    with np.errstate(invalid="ignore", divide="ignore"):
        assert np.isnan(mean[0]) and np.array_equal(mean[1:], s[1:] / n[1:])
        assert np.isnan(var[0]) and var[1] == 0.0 and np.array_equal(var[2:], m2[2:] / (n[2:] - 1))


WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
    import numpy as np, torch.distributed as dist
    from samsim_b200 import distributed as D
    from group_stats_ref import group_stats
    dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
    rank, world = dist.get_rank(), dist.get_world_size()
    z = np.load(%(data)r)
    X, Cm, goc, ngroup = z["X"], z["C"], z["goc"], int(z["ngroup"])
    col0, n = D.shard(len(goc), rank, world)
    R = 2   # two records: the second with other values
    st = np.stack([group_stats(X[r][col0:col0 + n], Cm[r][col0:col0 + n], goc[col0:col0 + n], ngroup) for r in range(R)])
    local = {"time": np.array([0.0, 10.0]), "i": np.array([1, 2]), "quantities": [("q", None)] * X.shape[2]}
    local.update({k: st[..., s] for s, k in enumerate(("count", "mean", "var", "min", "max"))})
    out = D.reduce_group_stats(local)
    if rank == 0:
        np.savez(%(out)r, **{k: out[k] for k in ("count", "mean", "var", "min", "max")})
    dist.destroy_process_group()
""")


def _data(ncol=600, Q=7, seed=6):
    rng = np.random.default_rng(seed)
    goc = rng.integers(0, 4, ncol).astype(np.int32)           # groups 0..3 span every shard boundary
    goc[:150] = 4                                            # group 4: only in the first shard
    goc[-120:] = 5                                           # group 5: only in the last shard
    goc[rng.random(ncol) < 0.05] = -1
    ngroup = 7                                               # group 6: empty everywhere
    X = rng.normal(5.0, 2.0, (2, ncol, Q)) * 10.0 ** rng.integers(-3, 4, (1, 1, Q))
    X[:, :, 0] = 3.25                                        # no spread: variance exactly 0
    Cm = rng.random((2, ncol, Q)) < 0.8
    Cm[:, goc == 3, 1] = False                               # a group without contributors in one quantity
    return X, Cm, goc, ngroup


@pytest.mark.parametrize("world", [2, 3])
def test_reduce_group_stats_gloo(tmp_path, world):
    X, Cm, goc, ngroup = _data()
    data = tmp_path / "data.npz"
    np.savez(data, X=X, C=Cm, goc=goc, ngroup=ngroup)
    out = tmp_path / "out.npz"
    script = tmp_path / "w.py"
    script.write_text(WORKER % {"root": str(ROOT), "tests": str(HERE), "data": str(data), "out": str(out)})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(29560 + world), WORLD_SIZE=str(world))
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r))) for r in range(world)]
    for p in procs:
        assert p.wait(timeout=300) == 0
    got = np.load(out)
    ref = np.stack([group_stats(X[r], Cm[r], goc, ngroup) for r in range(2)])
    cnt = ref[..., 0]
    assert np.array_equal(got["count"], cnt)
    for s, k in ((3, "min"), (4, "max")):
        assert np.array_equal(got[k], ref[..., s], equal_nan=True), k
    empty = cnt == 0
    assert empty[:, 6].all() and empty[:, 3, 1].all()
    assert np.isnan(got["mean"][empty]).all() and np.isnan(got["var"][empty]).all()
    m, v = ref[..., 1][~empty], ref[..., 2][~empty]
    assert np.allclose(got["mean"][~empty], m, rtol=1e-13, atol=0.0)
    assert (np.abs(got["var"][~empty] - v) <= np.maximum(1e-10 * np.abs(v), 1e-12 * m * m)).all()
    assert (got["var"][:, :6, 0] == 0.0).all()
