"""Test oracle of the all-contour distances (``contours="all"``; build-defined, no reference counterpart).

The vertex set of a class mask is every crack between 4-adjacent unequal pixels (``all_crack_vertices``, which
``test_oracle_contours.py::test_vertices_are_exactly_the_cracks`` proves equal to the union of all contours of the
restated ``find_contours``), each once, sorted into raster order of the doubled lattice.  Squared distances come from
an exact brute-force search for small sets and from ``scipy.ndimage.distance_transform_edt`` on the doubled lattice
(feature indices, exact integer arithmetic) for large ones.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

from oracle.contours_oracle import all_crack_vertices, directed_sq_distances

BRUTE_FORCE_MAX = 1 << 22        # |src| * |qry| up to which the brute-force search is used


def all_vertices(mask):
    """int64 (n, 2) doubled-lattice (y2, x2) vertices of every contour of ``mask``, raster order, each once."""
    v = all_crack_vertices(mask)
    return v[np.lexsort((v[:, 1], v[:, 0]))]


def edt_sq_distances(src, qry, shape):
    """For each vertex of ``qry`` the exact squared distance to the nearest vertex of ``src``, both on the doubled
    lattice of an image of ``shape`` (H, W): an EDT of the (2H - 1) x (2W - 1) grid whose zeros are ``src``."""
    h, w = shape
    grid = np.ones((2 * h - 1, 2 * w - 1), dtype=bool)
    grid[src[:, 0], src[:, 1]] = False
    idx = ndimage.distance_transform_edt(grid, return_distances=False, return_indices=True)
    ny = idx[0][qry[:, 0], qry[:, 1]].astype(np.int64)
    nx = idx[1][qry[:, 0], qry[:, 1]].astype(np.int64)
    return (ny - qry[:, 0]) ** 2 + (nx - qry[:, 1]) ** 2


def sq_distances(src, qry, shape):
    if len(src) * len(qry) <= BRUTE_FORCE_MAX:
        return directed_sq_distances(src, qry)
    return edt_sq_distances(src, qry, shape)


def all_contour_intermediates(mask_true, mask_pred):
    """Vertices and exact squared distances behind the all-contour hausdorff / hd95 / assd of one mask pair, or None
    when either set is empty (class absent from a map or filling it)."""
    mt, mp = np.asarray(mask_true), np.asarray(mask_pred)
    vt, vp = all_vertices(mt), all_vertices(mp)
    if len(vt) == 0 or len(vp) == 0:
        return None
    return {"verts_true": vt, "verts_pred": vp,
            "sq_pred_to_true": sq_distances(vt, vp, mt.shape),     # direction 0: every pred vertex -> true set
            "sq_true_to_pred": sq_distances(vp, vt, mt.shape)}     # direction 1: every true vertex -> pred set


def pack(v):
    """(n, 2) lattice vertices -> the library's packed uint32 ``y2 << 16 | x2``."""
    return (np.asarray(v, dtype=np.int64)[:, 0] << 16 | np.asarray(v, dtype=np.int64)[:, 1]).astype(np.uint32)
