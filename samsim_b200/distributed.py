"""Multi-GPU plumbing: one process per GPU, columns sharded, NO collective on the stepping path.

The only exchange SAMSIM-style ensembles need is the optional reduction / gather of diagnostics at output cadence
(SURVEY section 8e): 18 numbers per rank (sum/min/max of ice thickness, bulk salinity, freeboard, snow depth,
surface temperature, N_active) -> one all-reduce each for SUM / MIN / MAX over NCCL (gloo on CPU in the tests), and
the per-group statistics of the output records (reduce_group_stats) -> four all-reduces of [records, groups, quantities].
"""
from __future__ import annotations

import numpy as np

NAMES = ["thickness", "bulk_salin", "freeboard", "thick_snow", "T_top", "N_active"]


def shard(total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block of columns of `rank`: [col0, col0 + n); the remainder goes to the first ranks."""
    base, rem = divmod(total, world)
    n = base + (1 if rank < rem else 0)
    col0 = rank * base + min(rank, rem)
    return col0, n


def local_sites(site_of_col, col0: int, n: int) -> tuple[np.ndarray, np.ndarray]:
    """The forcing sites of the block [col0, col0 + n) of a rank: (sites, local_site_of_col).  `sites` are the
    sorted distinct sites the block reads and local_site_of_col[c] indexes into them, so the rank uploads
    table[sites] with local_site_of_col instead of the whole grid: table[sites][local_site_of_col] equals
    table[site_of_col[col0:col0 + n]]."""
    block = np.asarray(site_of_col)[col0:col0 + n]
    sites, local = np.unique(block, return_inverse=True)
    return sites, local.astype(np.int32).reshape(-1)


def reduce_ensemble(local: dict, ncol_local: int, group=None, device=None) -> dict:
    """local = Engine.reduce_diag() of this rank; returns the ensemble-wide mean/min/max per diagnostic."""
    import torch
    import torch.distributed as dist
    s = torch.tensor([local[n]["sum"] for n in NAMES] + [float(ncol_local)], dtype=torch.float64, device=device)
    mn = torch.tensor([local[n]["min"] for n in NAMES], dtype=torch.float64, device=device)
    mx = torch.tensor([local[n]["max"] for n in NAMES], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    total = float(s[-1].item())
    return {n: {"mean": float(s[j].item()) / total, "min": float(mn[j].item()), "max": float(mx[j].item())} for j, n in enumerate(NAMES)} | {"columns": int(total)}


def reduce_group_stats(local: dict, group=None, device=None) -> dict:
    """Combine Engine.group_stats() of ranks whose shards share column groups (same groups, depths, profiles and
    records on every rank; a group may be empty on some ranks).  All-reduces only: count and count*mean with SUM, then
    M2_r + n_r*(mean_r - mean)^2 with SUM, min / max with MIN / MAX.  Returns the same dict for the whole ensemble."""
    import torch
    import torch.distributed as dist
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    f64 = dict(dtype=torch.float64, device=device)
    n = torch.as_tensor(np.asarray(local["count"]), **f64)
    has = n > 0
    mean_r = torch.where(has, torch.as_tensor(np.asarray(local["mean"]), **f64), 0.0)
    sums = torch.stack([n, n * mean_r])
    if multi:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    N = sums[0]
    mean = sums[1] / N                                 # NaN where no rank has a contributor
    var_r = torch.as_tensor(np.asarray(local["var"]), **f64)
    m2 = torch.where(has, torch.where(n >= 2, var_r * (n - 1), 0.0) + n * (mean_r - mean) ** 2, 0.0)
    if multi:
        dist.all_reduce(m2, op=dist.ReduceOp.SUM, group=group)
    var = torch.where(N >= 2, m2 / (N - 1), torch.where(N == 1, 0.0, float("nan")))
    inf = float("inf")
    mn = torch.as_tensor(np.asarray(local["min"]), **f64)
    mx = torch.as_tensor(np.asarray(local["max"]), **f64)
    mn, mx = torch.where(mn.isnan(), inf, mn), torch.where(mx.isnan(), -inf, mx)
    if multi:
        dist.all_reduce(mn, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    nan = torch.full_like(N, float("nan"))
    out = {k: local[k] for k in ("time", "i", "quantities")}
    out.update(count=N.cpu().numpy(), mean=mean.cpu().numpy(), var=var.cpu().numpy(),
               min=torch.where(N > 0, mn, nan).cpu().numpy(), max=torch.where(N > 0, mx, nan).cpu().numpy())
    return out


def gather_columns(values, group=None, dst: int = 0):
    """Gather a per-column diagnostic (1-D tensor on this rank's device) to rank `dst` (None elsewhere)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return values
    world = dist.get_world_size(group)
    sizes = [torch.zeros(1, dtype=torch.int64, device=values.device) for _ in range(world)]
    dist.all_gather(sizes, torch.tensor([values.numel()], dtype=torch.int64, device=values.device), group=group)
    out = [torch.empty(int(sz.item()), dtype=values.dtype, device=values.device) for sz in sizes]
    dist.all_gather(out, values, group=group) if len({int(sz.item()) for sz in sizes}) == 1 else _uneven(out, values, group)
    return torch.cat(out) if dist.get_rank(group) == dst else None


def _uneven(out, values, group):
    import torch.distributed as dist
    for r, buf in enumerate(out):  # r = rank inside `group`; broadcast wants the GLOBAL rank of the source
        if r == dist.get_rank(group):
            buf.copy_(values)
        src = dist.get_global_rank(group, r) if group is not None else r
        dist.broadcast(buf, src=src, group=group)
