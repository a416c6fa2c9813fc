"""Test oracle of the full suite at any B-scan geometry: ``check_suite`` compares every integer and every contour
metric of one ``suite.evaluate(..., boundaries=True)`` result with the label-map oracle.

Contour ``[0]`` comes from the restated ``find_contours`` (``first_contour_lattice``); the nearest-vertex distances
come from a KD-tree, which only picks the index of a nearest vertex, and exact integer arithmetic, so that contours of
65k vertices stay affordable.  Results are cached per input item: one input checked under several seed policies, or
in a batch and alone, is scored once.
"""
from __future__ import annotations

import hashlib

import numpy as np
from scipy.spatial import cKDTree

from oracle import contours_oracle as co
from oracle import labelmap_oracle as lo

RTOL = 1e-6          # hd95 / assd: float64 epilogue against numpy's percentile and mean
SUM_RTOL = 1e-12     # sum of sqrt(D2 / 4): the kernels add in their own fixed order
INT_KEYS = ("confusion", "thickness_absdiff", "boundary_sq", "boundary_abs", "boundary_true", "boundary_pred")

_CACHE = {}


def nearest_sq(src, qry):
    """For each vertex of ``qry`` the exact squared distance (int64) to its nearest vertex of ``src``."""
    src = np.asarray(src, dtype=np.int64)
    qry = np.asarray(qry, dtype=np.int64)
    _, idx = cKDTree(src).query(qry)
    d = qry - src[idx]
    return (d * d).sum(axis=1)


def order_stats(sq):
    """max, the two neighbours of numpy's linear 95th percentile, and the float64 sum of sqrt(D2 / 4)."""
    s = np.sort(np.asarray(sq, dtype=np.int64))
    lo_i = int(np.floor((len(s) - 1) * 0.95))
    return int(s[-1]), (int(s[lo_i]), int(s[min(lo_i + 1, len(s) - 1)])), float(np.sqrt(s / 4.0).sum())


def contour_oracle(mask_true, mask_pred):
    """Contour ``[0]`` integers of one mask pair, or None when either mask has no contour: ``n_pts`` (true, pred),
    per direction (0: pred -> true, 1: true -> pred) ``max_sq``, ``p95`` and ``sum_dist``, and the reference's
    hausdorff / hd95 / assd from the exact squared distances."""
    try:
        vt = co.first_contour_lattice(mask_true)
        vp = co.first_contour_lattice(mask_pred)
    except IndexError:
        return None
    sq = (nearest_sq(vt, vp), nearest_sq(vp, vt))
    out = {"n_pts": (len(vt), len(vp)), "metrics": lo.contour_metrics_from_sq(*sq)}
    for d in (0, 1):
        out[d] = order_stats(sq[d])
    return out


def _key(a):
    a = np.ascontiguousarray(a)
    return a.shape, hashlib.blake2b(a.tobytes(), digest_size=16).hexdigest()


def item_oracle(yt, yp, k):
    """Oracle of one (H, W) item pair: ``score_bscan_fast`` integers and ``contour_oracle`` of every class (cached)."""
    key = (_key(yt), _key(yp), int(k))
    ref = _CACHE.get(key)
    if ref is None:
        ref = {"fast": lo.score_bscan_fast(yt, yp, k), "contours": [contour_oracle(yt == c, yp == c) for c in range(k)]}
        _CACHE[key] = ref
    return ref


def max_sq(yt, yp, k):
    """Largest contour ``[0]`` squared distance of an item over all classes and both directions (0 without contours)."""
    refs = [r for r in item_oracle(yt, yp, k)["contours"] if r is not None]
    return max([max(r[0][0], r[1][0]) for r in refs], default=0)


def check_suite(yt, yp, k, res, items=None):
    """``res`` (``suite.evaluate(..., boundaries=True)``) against the oracle.  ``yt`` / ``yp``: host ``[n, H, W]``;
    result item ``items[j]`` (default ``j``) is compared with ``yt[j]`` / ``yp[j]``.  Integers are exact, sum_dist
    within 1e-12, hausdorff bit-exact, hd95 and assd within 1e-6.  Returns the number of contour pairs compared."""
    ints, m = res.integers(), res.metrics()
    items = range(len(yt)) if items is None else items
    n_contours = 0
    for j, i in enumerate(items):
        ref = item_oracle(yt[j], yp[j], k)
        for key in INT_KEYS:
            assert np.array_equal(ints[key][i], ref["fast"][key]), (i, key)
        for c in range(k):
            r = ref["contours"][c]
            where = (i, c)
            if r is None:
                assert ints["contour_n_pts"][i, c, 0] == 0 or ints["contour_n_pts"][i, c, 1] == 0, where
                assert np.isnan(m["hausdorff_distance"][i, c]), where
                continue
            n_contours += 1
            assert tuple(int(v) for v in ints["contour_n_pts"][i, c]) == r["n_pts"], (where, ints["contour_n_pts"][i, c])
            for d in (0, 1):
                vmax, p95, dsum = r[d]
                assert ints["contour_max_sq"][i, c, d] == vmax, (where, d, ints["contour_max_sq"][i, c, d], vmax)
                assert tuple(int(v) for v in ints["contour_p95_sq"][i, c, d]) == p95, (where, d)
                np.testing.assert_allclose(ints["contour_sum_dist"][i, c, d], dsum, rtol=SUM_RTOL, err_msg=str((where, d)))
            rm = r["metrics"]
            assert m["hausdorff_distance"][i, c] == rm["hausdorff_distance"], where
            np.testing.assert_allclose(m["hausdorff_distance_95"][i, c], rm["hausdorff_distance_95"], rtol=RTOL,
                                       err_msg=str(where))
            np.testing.assert_allclose(m["assd"][i, c], rm["assd"], rtol=RTOL, err_msg=str(where))
    return n_contours


def sawtooth_pair(h, w, n_vertices, shift):
    """A 2-class layered pair (class 0 above a boundary row b(x), class 1 from it down) whose boundary zig-zags so that
    contour ``[0]`` of class 0 has exactly ``n_vertices`` = W + sum |b(x + 1) - b(x)| vertices: one vertical crack per
    column, one horizontal crack per row crossed between columns.  The prediction is the same boundary ``shift`` rows
    lower.  Returns ``uint8 [1, h, w]`` arrays."""
    total = int(n_vertices) - int(w)
    steps = w - 1
    if total < 0 or steps <= 0:
        raise ValueError("n_vertices must be at least W, and W at least 2")
    d = np.full(steps, total // steps, dtype=np.int64)
    d[:total % steps] += 1                                   # sum(d) == total
    top = int(d.max())
    base = (h - top - abs(int(shift))) // 2
    if base < 1 or base + top + abs(int(shift)) > h - 1:
        raise ValueError(f"{n_vertices} vertices do not fit a {h}x{w} map")
    b = np.empty(w, dtype=np.int64)
    b[0] = base
    for x in range(steps):                                    # up by d[x] from the base, back down by the next step
        b[x + 1] = base + d[x] if b[x] == base else b[x] - d[x]
        if b[x + 1] < base:                                   # a longer step down than up: go back up instead
            b[x + 1] = b[x] + d[x]
    assert np.abs(np.diff(b)).sum() == total and b.min() >= 1 and b.max() + abs(int(shift)) <= h - 1
    y = np.arange(h)[:, None]
    yt = (y >= b[None, :]).astype(np.uint8)
    yp = (y >= b[None, :] + int(shift)).astype(np.uint8)
    return yt[None], yp[None]
