"""Multi-GPU sharding: one process per GPU, B-scans partitioned contiguously, ONE small all-reduce.

Every reference function is a pure function of one (y_true, y_pred) pair, so items shard with no
data-path collective (SURVEY.md 8e).  What crosses NVLink is a packed float64 vector of a few
hundred bytes per rank: summed confusion counts, column-scan sums, per-class sums of the contour
metrics and their valid-item counts.  Integer partials ride in float64 exactly (each must stay
below 2**53, which is checked), so the totals are identical for every world size; the genuine
floating-point sums differ by rounding only (<= 1e-12 relative).  ``want_max=True`` adds a second
(MAX) all-reduce for the dataset-level Hausdorff maximum.
"""
from __future__ import annotations

import numpy as np

from . import derive

_EXACT_LIMIT = float(2 ** 53)


def shard_range(n_items, rank, world):
    """Contiguous [start, stop) of the items rank `rank` scores; sizes differ by at most one."""
    base, rem = divmod(n_items, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def local_partials(ints, metrics, num_classes):
    """Pack this rank's sums into one float64 vector (layout mirrored by ``unpack`` and by the device-side
    ``totals_kernel``: the SUM-reducible head of ``octm_derive_metrics``' totals)."""
    k = num_classes
    parts = [np.asarray([ints["confusion"].shape[0]], np.float64),
             ints["confusion"].astype(np.int64).sum(0).reshape(-1).astype(np.float64)]
    if "thickness_absdiff" in ints:
        parts += [ints["thickness_absdiff"].sum(0).astype(np.float64),
                  ints["boundary_sq"].sum(0).astype(np.float64), ints["boundary_abs"].sum(0).astype(np.float64)]
    else:
        parts += [np.zeros(k), np.zeros(k - 1), np.zeros(k - 1)]
    if "contour_valid" in metrics:
        valid = metrics["contour_valid"]
        parts.append(valid.sum(0).astype(np.float64))
        for name in ("hausdorff_distance", "hausdorff_distance_95", "assd"):
            parts.append(np.where(valid, metrics[name], 0.0).sum(0))
    else:
        parts += [np.zeros(k)] * 4
    n_over = 0
    if "contour_flags" in ints:
        n_over = int(((np.asarray(ints["contour_flags"]).astype(np.int64) & 12) != 0).any(axis=1).sum())
    n_bad = 0
    if "item_pixels" in ints:
        cm = ints["confusion"].astype(np.int64)
        n_bad = int((cm.reshape(cm.shape[0], -1).sum(1) != int(ints["item_pixels"])).sum())
    parts.append(np.asarray([n_over, n_bad], np.float64))
    vec = np.concatenate(parts)
    _check_exact(vec, k)
    return vec


def _check_exact(vec, k):
    n_exact = 1 + k * k + k + 2 * (k - 1) + k
    if np.any(np.abs(vec[:n_exact]) >= _EXACT_LIMIT):
        raise OverflowError("an integer partial exceeds 2**53 and would not be exact in the float64 all-reduce")


def unpack(vec, num_classes, width):
    k = num_classes
    o = 0

    def take(m):
        nonlocal o
        out = vec[o:o + m]
        o += m
        return out

    n_items = int(round(take(1)[0]))
    cm = np.rint(take(k * k)).astype(np.int64).reshape(k, k)
    thick = np.rint(take(k)).astype(np.int64)
    bsq, bab = np.rint(take(k - 1)).astype(np.int64), np.rint(take(k - 1)).astype(np.int64)
    nvalid = np.rint(take(k)).astype(np.int64)
    s_hd, s_hd95, s_assd = take(k), take(k), take(k)
    n_over, n_bad = (int(round(x)) for x in take(2))
    out = {"n_items": n_items, "confusion": cm, "contour_items": nvalid, "n_overflow_items": n_over,
           "n_bad_label_items": n_bad}
    out.update(derive.count_metrics(*derive.class_counts(cm)))          # pooled (micro) ratios per class
    denom = max(n_items, 1) * width
    out["thickness_difference"] = thick.astype(np.float64) / denom       # mean over all columns of all items
    out["boundary_mse"] = bsq.astype(np.float64) / denom
    out["boundary_rmse"] = np.sqrt(out["boundary_mse"])
    out["boundary_mad"] = bab.astype(np.float64) / denom
    with np.errstate(invalid="ignore", divide="ignore"):
        out["hausdorff_distance_mean"] = s_hd / nvalid
        out["hausdorff_distance_95_mean"] = s_hd95 / nvalid
        out["assd_mean"] = s_assd / nvalid
    return out


def all_reduce_sum(vec, world, device=None, group=None):
    """float64 SUM all-reduce of a small numpy vector (NCCL on `device`, gloo when device is None/cpu)."""
    if world == 1:
        return vec
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(vec))
    if device is not None and str(device) != "cpu":
        t = t.to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


def base_len(num_classes):
    """Length of the SUM-reducible head of the totals vector (``octm_totals_sum_len``)."""
    k = num_classes
    return 1 + k * k + k + 2 * (k - 1) + 4 * k + 2


def _enqueue_reduce(res, world, group, want_max):
    """(local, reduced) vectors: ``reduced`` = totals summed (head) / maximised (Hausdorff maxima) over the
    ranks, enqueued on the current stream for CUDA totals.  No host round trip."""
    k = res.labels.num_classes
    nb = base_len(k)
    local = res.totals
    reduced = local.clone()
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(reduced[:nb], op=dist.ReduceOp.SUM, group=group)
        if want_max:
            dist.all_reduce(reduced[nb:nb + k], op=dist.ReduceOp.MAX, group=group)
    return local, reduced


def _finish(res, world, group, want_max, local, reduced):
    """Read the reduced totals back (one small D2H) and take the decisions EVERY rank must take alike, from the
    REDUCED vector: ``n_bad_label_items > 0`` raises ValueError on all ranks; ``n_overflow_items > 0`` (a contour
    longer than max_pts on ANY rank) makes every rank settle its own overflowed items and join a second
    reduction.  Deciding from the local flags would leave the other ranks outside the second collective."""
    import torch
    k, w = res.labels.num_classes, res.labels.width
    nb = base_len(k)
    for attempt in range(2):
        both = torch.stack([local, reduced]).cpu().numpy()              # one D2H
        vec_local, vec = both[0], both[1]
        if int(round(vec[nb - 1])) > 0 and res.validate:
            res._totals_host, res._final, res._inputs = vec_local, True, None
            raise ValueError(f"{int(round(vec[nb - 1]))} item(s) hold a label >= num_classes {k}")
        if int(round(vec[nb - 2])) > 0 and attempt == 0 and res.contours is not None:
            res.settle_overflow(vec_local)                               # local redo (no-op on ranks without overflow)
            local, reduced = _enqueue_reduce(res, world, group, want_max)
            continue
        break
    if res._totals_host is None:
        res._totals_host, res._final, res._inputs = vec_local, True, None
    _check_exact(vec_local, k)
    out = unpack(vec[:nb], k, w)
    if want_max:
        out["hausdorff_distance_max"] = np.where(vec[nb:nb + k] < 0, np.nan, vec[nb:nb + k])
    return out


def dataset_totals(res, world, device=None, group=None, want_max=False):
    """Dataset-level numbers over all ranks' shards from one SuiteResult per rank.

    The per-rank partial sums come from the device-side totals kernel and are summed across ranks by ONE
    float64 all-reduce issued directly on the device vector (stream ordered after the kernels, no host round
    trip before the collective); a single small D2H then brings the reduced sums and this rank's own vector
    to the host.  Contour-overflow retries and the invalid-label error are decided from the reduced vector,
    i.e. collectively (see ``_finish``)."""
    local, reduced = _enqueue_reduce(res, world, group, want_max)
    return _finish(res, world, group, want_max, local, reduced)


class PendingTotals:
    """Dataset totals whose device work (totals kernel, all-reduce) is enqueued but not yet read back."""

    def __init__(self, res, world, group, want_max, local, reduced):
        self.res, self.world, self.group, self.want_max = res, world, group, want_max
        self.local, self.reduced = local, reduced

    def result(self):
        """One small D2H; overflow retries are collective (every rank re-reduces when any rank overflowed)."""
        return _finish(self.res, self.world, self.group, self.want_max, self.local, self.reduced)


def dataset_totals_async(res, world, group=None, want_max=False):
    """Enqueue the cross-rank reduction of ``res.totals`` on the current stream and return a
    ``PendingTotals``; nothing is copied to the host until ``.result()``.  Lets a caller keep several
    evaluations in flight (the benchmark's device-timed region does)."""
    local, reduced = _enqueue_reduce(res, world, group, want_max)
    return PendingTotals(res, world, group, want_max, local, reduced)


def surface_dice_totals(res, world, device=None, group=None):
    """Dataset-level normalized surface Dice over all ranks' shards from one ``evaluate(surface_dice=...)`` result per
    rank: per class and tolerance, ``surface_dice_mean`` = mean over the items where NSD is defined (as
    ``hausdorff_distance_mean``) and ``surface_dice_items`` = their exact count, both ``[K, T]``.  One float64 SUM
    all-reduce of its own small vector; the totals vector of ``dataset_totals`` is not touched."""
    taus = res.surface_dice_tolerances
    if taus is None:
        raise ValueError("the result has no surface Dice counts: evaluate with surface_dice=...")
    ints = res.integers()
    nsd = derive.surface_dice(ints["surface_dice_n_surf"], ints["surface_dice_n_within"])      # [N, K, T]
    defined = ~np.isnan(nsd)
    vec = np.concatenate([defined.sum(0).reshape(-1).astype(np.float64), np.where(defined, nsd, 0.0).sum(0).reshape(-1)])
    vec = all_reduce_sum(vec, world, device=device, group=group)
    k, t = nsd.shape[1:]
    items = np.rint(vec[:k * t]).astype(np.int64).reshape(k, t)
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = vec[k * t:].reshape(k, t) / items
    return {"surface_dice_mean": mean, "surface_dice_items": items, "tolerances": tuple(taus)}


def component_totals(res, world, device=None, group=None):
    """Dataset-level component scores over all ranks' shards from one ``evaluate(components=4 or 8)`` result per rank.
    The counts of every item are summed (one float64 SUM all-reduce of its own small vector; each sum is exact below
    2**53, and the totals vector of ``dataset_totals`` is not touched).  Per class: pooled (micro) ``component_recall``,
    ``component_precision`` and ``component_f1`` by the rules of ``derive.component_metrics`` applied to the summed
    counts, ``component_count_error`` = the mean of |n_t - n_p| over all items, and the summed integers
    ``component_count`` / ``component_hits`` ``[K, 2]`` and ``items``."""
    if res.component_connectivity is None:
        raise ValueError("the result has no component counts: evaluate with components=4 or 8")
    ints = res.integers()
    nc = ints["component_count"].astype(np.int64)                 # [N, K, 2]
    nh = ints["component_hits"].astype(np.int64)
    err = np.abs(nc[..., 0] - nc[..., 1]).sum(0)
    vec = np.concatenate([nc.sum(0).reshape(-1), nh.sum(0).reshape(-1), err, [nc.shape[0]]]).astype(np.float64)
    vec = all_reduce_sum(vec, world, device=device, group=group)
    k = nc.shape[1]
    tot = np.rint(vec).astype(np.int64)
    count, hits = tot[:2 * k].reshape(k, 2), tot[2 * k:4 * k].reshape(k, 2)
    items = int(tot[-1])
    out = derive.component_metrics(count, hits)
    with np.errstate(invalid="ignore", divide="ignore"):
        out["component_count_error"] = tot[4 * k:5 * k] / np.float64(items) if items else np.full(k, np.nan)
    out.update(component_count=count, component_hits=hits, items=items, connectivity=res.component_connectivity)
    return out


def surface_distance_3d_sharded(vol_true, vol_pred, num_classes, rank, world, group=None):
    """BASELINE config 5 on several GPUs: the volume pair is replicated (it is small), the ``2 * K``
    independent (class, direction) distance transforms are split into contiguous unit ranges per rank,
    and the per-unit integers / sums are combined by ONE small all-reduce (every unit is written by exactly
    one rank, the others contribute zeros, so the sum is exact).  Returns the same dict as
    ``suite.surface_distance_3d`` with identical contents on every rank."""
    import torch
    from . import suite
    ub, ue = shard_range(2 * num_classes, rank, world)
    ints = suite.surface_distance_3d(vol_true, vol_pred, num_classes, units=(ub, ue))
    if world > 1:
        import torch.distributed as dist
        packed = torch.cat([ints["n_pts"].to(torch.float64).reshape(-1), ints["max_sq"].to(torch.float64).reshape(-1),
                            ints["p95_sq"].to(torch.float64).reshape(-1), ints["sum_dist"].reshape(-1)])
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
        k = num_classes
        o = 0
        for key, shape, dt in (("n_pts", (k, 2), torch.int32), ("max_sq", (k, 2), torch.int32),
                               ("p95_sq", (k, 2, 2), torch.int32), ("sum_dist", (k, 2), torch.float64)):
            m = int(np.prod(shape))
            v = packed[o:o + m].reshape(shape)
            ints[key] = v.to(torch.int64).to(dt) if dt != torch.float64 else v.clone()
            o += m
    return ints
