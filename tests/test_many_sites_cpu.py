"""distributed.local_sites: each rank uploads only the forcing sites its block of columns reads."""
import numpy as np
import pytest

from samsim_b200 import distributed as D


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("nsite", [1, 7, 500])
def test_local_sites_reproduce_the_global_table(world, nsite):
    rng = np.random.default_rng(world * 1000 + nsite)
    ncol = 1001
    table = rng.normal(size=(nsite, 4, 5))
    site_of_col = rng.integers(0, nsite, ncol).astype(np.int32)
    covered = np.zeros(ncol, dtype=int)
    for rank in range(world):
        col0, n = D.shard(ncol, rank, world)
        sites, local = D.local_sites(site_of_col, col0, n)
        assert local.dtype == np.int32 and local.shape == (n,)
        assert (np.diff(sites) > 0).all() and set(sites) == set(site_of_col[col0:col0 + n])
        assert np.array_equal(table[sites][local], table[site_of_col[col0:col0 + n]])
        covered[col0:col0 + n] += 1
    assert (covered == 1).all()
