"""Test oracle of the B-scan contour distances with a pixel spacing ``(sy, sx)`` (rows, columns).

The vertex sets are those of the existing oracles: contour ``[0]`` of ``find_contours`` (``first_contour_lattice``, with
its closing repeat) and every crack of the class mask (``all_contours_oracle.all_vertices``).  A vertex pair at lattice
offset (a, b) is ``q = fl(fl(wy * a**2) + fl(wx * b**2))`` with ``wy = sy * sy`` and ``wx = sx * sx`` in float64; a query's
``d2`` is the minimum of ``q`` over the source set (brute force), its distance ``sqrt(d2 / 4.0)``.
"""
from __future__ import annotations

import math

import numpy as np

from oracle.contours_oracle import first_contour_lattice
from all_contours_oracle import all_vertices


def weights(spacing):
    sy, sx = (float(v) for v in spacing)
    return sy * sy, sx * sx


def q_of_offsets(a, b, spacing):
    """``q`` of lattice offsets (arrays of equal shape), float64, in the contract's order of operations."""
    wy, wx = weights(spacing)
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return wy * (a * a) + wx * (b * b)


def squared_distances(src, qry, spacing):
    """For each vertex of ``qry`` the minimum ``q`` to ``src`` (both (n, 2) int lattice vertices), float64."""
    src = np.asarray(src, dtype=np.int64)
    qry = np.asarray(qry, dtype=np.int64)
    out = np.empty(len(qry), dtype=np.float64)
    step = max(1, (1 << 22) // max(1, len(src)))
    for s in range(0, len(qry), step):
        q = qry[s:s + step]
        out[s:s + step] = q_of_offsets(q[:, None, 0] - src[None, :, 0], q[:, None, 1] - src[None, :, 1], spacing).min(1)
    return out


def python_search(src, qry, spacing):
    """The same minimum in plain Python floats, one pair at a time (the cross-check of ``squared_distances``)."""
    wy, wx = weights(spacing)
    out = []
    for qy, qx in qry:
        best = math.inf
        for sy, sx in src:
            a, b = int(qy) - int(sy), int(qx) - int(sx)
            best = min(best, wy * float(a * a) + wx * float(b * b))
        out.append(best)
    return np.asarray(out, dtype=np.float64)


def vertices(mask, mode):
    """Lattice vertices of ``mask`` in contour mode ``"first"`` (contour [0]) or ``"all"``; None when there are none."""
    if mode == "first":
        try:
            return first_contour_lattice(np.asarray(mask))
        except IndexError:
            return None
    v = all_vertices(np.asarray(mask))
    return v if len(v) else None


def intermediates(mask_true, mask_pred, spacing, mode="all"):
    """Vertices and float64 ``d2`` of both directions for one mask pair, or None when either set is empty."""
    vt, vp = vertices(mask_true, mode), vertices(mask_pred, mode)
    if vt is None or vp is None:
        return None
    return {"verts_true": vt, "verts_pred": vp,
            "sq_pred_to_true": squared_distances(vt, vp, spacing),     # direction 0
            "sq_true_to_pred": squared_distances(vp, vt, spacing)}     # direction 1


def order_statistics(d2):
    """(max, the d2 of rank floor((m - 1) * 0.95), the next one or the same at the end) of one direction."""
    s = np.sort(np.asarray(d2, dtype=np.float64))
    m = len(s)
    lo = int(np.floor((m - 1) * 0.95))
    return s[-1], s[lo], s[min(lo + 1, m - 1)]


def surface_dice_counts(mask_true, mask_pred, spacing, taus):
    """(n_surf (|V_t|, |V_p|), n_within [2][T]) of the all-contour sets: a query is within tau when sqrt(d2 / 4.0) <= tau."""
    vt, vp = vertices(mask_true, "all"), vertices(mask_pred, "all")
    n_surf = (0 if vt is None else len(vt), 0 if vp is None else len(vp))
    n_within = np.zeros((2, len(taus)), dtype=np.int64)
    if vt is not None and vp is not None:
        for d, (src, qry) in enumerate(((vt, vp), (vp, vt))):
            dist = np.sqrt(squared_distances(src, qry, spacing) / 4.0)
            for j, tau in enumerate(taus):
                n_within[d, j] = int((dist <= tau).sum())
    return n_surf, n_within
