"""Test oracle of the normalized surface Dice (``surface_dice=``; build-defined, no reference counterpart).

The surfaces are the all-contour vertex sets of ``all_contours_oracle`` and the squared distances its exact nearest
vertex searches (brute force or EDT).  A vertex counts as within ``tau`` when ``np.sqrt(sq / 4.0) <= tau``: the public
definition taken literally, not the integer threshold the library derives from it.
"""
from __future__ import annotations

import numpy as np

from all_contours_oracle import all_vertices, sq_distances


def mask_counts(mask_true, mask_pred, taus):
    """``n_surf (2,)`` = (|V_t|, |V_p|) and ``n_within (2, T)`` (direction 0: pred vertices within tau of the true
    boundary, 1: the other way) of one mask pair."""
    mt, mp = np.asarray(mask_true), np.asarray(mask_pred)
    vt, vp = all_vertices(mt), all_vertices(mp)
    n_surf = np.array([len(vt), len(vp)], dtype=np.int64)
    n_within = np.zeros((2, len(taus)), dtype=np.int64)
    if len(vt) and len(vp):
        for d, sq in enumerate((sq_distances(vt, vp, mt.shape), sq_distances(vp, vt, mt.shape))):
            dist = np.sqrt(sq / 4.0)
            n_within[d] = [int(np.count_nonzero(dist <= t)) for t in taus]
    return n_surf, n_within


def label_counts(yt, yp, num_classes, taus):
    """``n_surf [N, K, 2]`` and ``n_within [N, K, 2, T]`` of label maps ``[N, H, W]``."""
    n = yt.shape[0]
    ns = np.zeros((n, num_classes, 2), dtype=np.int64)
    nw = np.zeros((n, num_classes, 2, len(taus)), dtype=np.int64)
    for i in range(n):
        for c in range(num_classes):
            ns[i, c], nw[i, c] = mask_counts(yt[i] == c, yp[i] == c, taus)
    return ns, nw
