"""Fast exact oracles of the optional passes (``contours="all"``, ``spacing=``, ``surface_dice=``, ``components=``) at
the geometry envelope, where the brute-force oracles would compare ~30k x 30k vertex pairs per class.

* All-contour squared distances: a KD-tree picks the index of a nearest vertex, exact int64 arithmetic gives its D2
  (``geometry_oracle.nearest_sq``) on the vertex sets of ``all_contours_oracle.all_vertices``.
* Squared distances with a spacing ``(sy, sx)``: a KD-tree on ``(sy * y2, sx * x2)`` gives the nearest distance r of
  each query, then every source vertex within ``r * (1 + 1e-9)`` is a candidate and the query's ``d2`` is the minimum
  of the contract's ``q = fl(fl(wy * a**2) + fl(wx * b**2))`` over them.  The vertex that minimises ``q`` lies at a
  real distance within a few float64 roundings of r, far inside the ball, so the minimum is the brute-force one.
* Surface Dice counts: from those distances, ``sqrt(d / 4.0) <= tau``, as ``surface_dice_oracle`` counts them.
* Component counts: ``components_oracle`` (scipy.ndimage.label), already fast.

Results are cached per input item, so an item checked in a batch, alone and under several options is scored once.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

import components_oracle as cco
import spacing_2d_oracle as so
from geometry_oracle import _key, nearest_sq

BALL = 1.0 + 1e-9          # candidate radius over the KD-tree's nearest distance

_CACHE = {}


def spacing_d2(src, qry, spacing):
    """For each vertex of ``qry`` the minimum float64 ``q`` to ``src`` (both (n, 2) int lattice vertices), exactly
    ``spacing_2d_oracle.squared_distances``."""
    src = np.asarray(src, dtype=np.int64)
    qry = np.asarray(qry, dtype=np.int64)
    sy, sx = (float(v) for v in spacing)
    scale = np.array([sy, sx])
    tree = cKDTree(src * scale)
    pts = qry * scale
    r, _ = tree.query(pts, workers=-1)
    cand = tree.query_ball_point(pts, r * BALL, workers=-1, return_sorted=False)
    lens = np.fromiter((len(c) for c in cand), dtype=np.int64, count=len(cand))
    assert (lens > 0).all()
    idx = np.concatenate([np.asarray(c, dtype=np.int64) for c in cand])
    qi = np.repeat(np.arange(len(qry)), lens)
    q = so.q_of_offsets(qry[qi, 0] - src[idx, 0], qry[qi, 1] - src[idx, 1], spacing)
    return np.minimum.reduceat(q, np.concatenate([[0], np.cumsum(lens)[:-1]]))


def distances(src, qry, spacing=None):
    """Exact nearest-vertex squared distances: int64 D2 in pixels, float64 ``q`` with a spacing."""
    return nearest_sq(src, qry) if spacing is None else spacing_d2(src, qry, spacing)


def order_stats(d):
    """(max, the d of rank floor((m - 1) * 0.95), the next one or the same at the end, sum of sqrt(d / 4.0))."""
    s = np.sort(np.asarray(d))
    lo = int(np.floor((len(s) - 1) * 0.95))
    return s[-1], s[lo], s[min(lo + 1, len(s) - 1)], float(np.sqrt(s / 4.0).sum())


def _vertices(mask, mode):
    v = so.vertices(mask, mode)
    return np.zeros((0, 2), np.int64) if v is None else np.asarray(v, dtype=np.int64)


def contours(yt, yp, k, mode="all", spacing=None):
    """Per class of one (H, W) item pair: ``(vt, vp, d)`` with the vertex sets of ``mode`` (``"all"``: every crack,
    raster order; ``"first"``: contour [0] with its closing repeat) and ``d = (pred -> true, true -> pred)``
    distances, ``d = None`` when either set is empty (cached)."""
    key = ("contours", _key(yt), _key(yp), int(k), mode, None if spacing is None else tuple(float(v) for v in spacing))
    ref = _CACHE.get(key)
    if ref is None:
        ref = []
        for c in range(k):
            vt, vp = _vertices(yt == c, mode), _vertices(yp == c, mode)
            d = None
            if len(vt) and len(vp):
                d = (distances(vt, vp, spacing), distances(vp, vt, spacing))
            ref.append((vt, vp, d))
        _CACHE[key] = ref
    return ref


def surface_counts(yt, yp, k, taus, spacing=None):
    """``n_surf [K, 2]`` (|V_t|, |V_p|) and ``n_within [K, 2, T]`` of one item pair: direction 0 counts the pred
    vertices within tau of the true boundary, 1 the other way; within means ``sqrt(d / 4.0) <= tau``."""
    n_surf = np.zeros((k, 2), np.int64)
    n_within = np.zeros((k, 2, len(taus)), np.int64)
    for c, (vt, vp, d) in enumerate(contours(yt, yp, k, "all", spacing)):
        n_surf[c] = len(vt), len(vp)
        if d is not None:
            for di in (0, 1):
                dist = np.sqrt(d[di] / 4.0)
                n_within[c, di] = [int(np.count_nonzero(dist <= t)) for t in taus]
    return n_surf, n_within


def component_counts(yt, yp, k, connectivity):
    """``n_comp [K, 2]`` and ``n_hit [K, 2]`` of one item pair (cached)."""
    key = ("components", _key(yt), _key(yp), int(k), int(connectivity))
    ref = _CACHE.get(key)
    if ref is None:
        nc, nh = cco.label_counts(np.asarray(yt)[None], np.asarray(yp)[None], k, connectivity)
        ref = _CACHE[key] = (nc[0], nh[0])
    return ref

