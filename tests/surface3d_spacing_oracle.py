"""Test oracle of the 3-D surface distances with a voxel spacing and of the volumetric normalized surface Dice
(``suite.surface_distance_3d(spacing=..., tolerances=...)``; build-defined, pinned to scipy).

Surfaces are those of ``oracle/surface3d_oracle.py`` (``mask & ~binary_erosion(mask)``).  The nearest source voxel of
every query voxel is scipy's (``distance_transform_edt(~surface, sampling=spacing, return_indices=True)``); its squared
distance is then computed from the integer offset (a, b, c) by the library's definition, in float64 and in this order:

    d2 = w0 * a**2 + (w1 * b**2 + w2 * c**2),        w_i = spacing[i] ** 2

A query voxel is within ``tau`` when ``np.sqrt(d2) <= tau``.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

from oracle.surface3d_oracle import surface


def weights(spacing):
    return tuple(float(s) * float(s) for s in spacing)


def d2_of_offsets(off, spacing):
    """float64 squared distances of integer offsets ``off [n, 3]`` by the library's expression."""
    w0, w1, w2 = weights(spacing)
    off = np.asarray(off, dtype=np.int64)
    a2, b2, c2 = (off[:, i] * off[:, i] for i in range(3))
    return w0 * a2 + (w1 * b2 + w2 * c2)


def squared_distances(mask_from, mask_to, spacing):
    """float64 squared distances from every surface voxel of ``mask_from`` (C order) to the nearest surface voxel of
    ``mask_to`` (None when either surface is empty)."""
    sa, sb = surface(mask_from), surface(mask_to)
    if not sa.any() or not sb.any():
        return None
    _, idx = ndimage.distance_transform_edt(~sb, sampling=tuple(float(s) for s in spacing), return_indices=True)
    q = np.argwhere(sa)
    return d2_of_offsets(q - idx[:, sa].T, spacing)


def class_metrics(vol_true, vol_pred, cls, spacing, taus=()):
    """Per class: the two lists of squared distances (direction 0: y_pred surface -> y_true surface), hd / hd95 / assd
    (NaN when either surface is empty), ``n_surf (2,)`` = (|S_t|, |S_p|), ``n_within (2, T)`` and the surface Dice."""
    mt, mp = vol_true == cls, vol_pred == cls
    d1 = squared_distances(mp, mt, spacing)
    d2 = squared_distances(mt, mp, spacing)
    n_surf = np.array([surface(mt).sum(), surface(mp).sum()], dtype=np.int64)
    n_within = np.zeros((2, len(taus)), dtype=np.int64)
    out = {"sq_pred_to_true": d1, "sq_true_to_pred": d2, "n_surf": n_surf, "n_within": n_within,
           "hausdorff_distance": np.nan, "hausdorff_distance_95": np.nan, "assd": np.nan}
    if d1 is not None and d2 is not None:
        e1, e2 = np.sqrt(d1), np.sqrt(d2)
        for d, e in enumerate((e1, e2)):
            n_within[d] = [int(np.count_nonzero(e <= t)) for t in taus]
        out.update(hausdorff_distance=max(e1.max(), e2.max()),
                   hausdorff_distance_95=max(np.percentile(e1, 95), np.percentile(e2, 95)),
                   assd=(np.mean(e1) + np.mean(e2)) / 2)
    tot = n_surf.sum()
    out["surface_dice"] = (n_within.sum(0) / tot) if tot else np.full(len(taus), np.nan)
    return out
