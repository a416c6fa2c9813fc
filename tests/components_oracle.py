"""Test oracle of the connected-component counts (``components=``; build-defined, no reference counterpart).

``n_comp[i, c, m]`` is ``scipy.ndimage.label(L_m == c, generate_binary_structure(2, 1 or 2))[1]`` and ``n_hit[i, c, m]``
the number of those labels found under ``(L_m == c) & (L_o == c)``: the public definition taken literally.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage


def structure(connectivity):
    return ndimage.generate_binary_structure(2, 1 if connectivity == 4 else 2)


def mask_counts(mask, other, connectivity):
    """(components of ``mask``, how many of them meet ``other``) of one binary mask pair."""
    lab, n = ndimage.label(np.asarray(mask, bool), structure(connectivity))
    hit = np.unique(lab[np.asarray(mask, bool) & np.asarray(other, bool)])
    return n, int(np.count_nonzero(hit))


def label_counts(yt, yp, num_classes, connectivity):
    """``n_comp [N, K, 2]`` and ``n_hit [N, K, 2]`` of label maps ``[N, H, W]`` (map 0: y_true, 1: y_pred)."""
    n = yt.shape[0]
    nc = np.zeros((n, num_classes, 2), dtype=np.int64)
    nh = np.zeros((n, num_classes, 2), dtype=np.int64)
    for i in range(n):
        for c in range(num_classes):
            mt, mp = yt[i] == c, yp[i] == c
            nc[i, c, 0], nh[i, c, 0] = mask_counts(mt, mp, connectivity)
            nc[i, c, 1], nh[i, c, 1] = mask_counts(mp, mt, connectivity)
    return nc, nh
