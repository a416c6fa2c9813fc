"""Oracle of the per-sector layer thickness (``suite.sector_thickness``, ``octm_sector_thickness_i32``): group thickness
from ``oracle.labelmap_oracle.column_thickness`` (pixels of each class per column), summed per region with
``np.add.at``.  ``python_sums`` is the same thing as a plain loop over A-scans, to check this one."""
import numpy as np

from oracle.labelmap_oracle import column_thickness


def group_thickness(label_map, num_classes, groups):
    """int64 [G, W]: pixels of the classes first .. last in every column of one (H, W) B-scan."""
    ct = column_thickness(label_map, num_classes)
    return np.stack([ct[f:last + 1].sum(axis=0) for f, last in groups])


def sector_sums(y_true, y_pred, num_classes, groups, regions, n_regions):
    """``y_true`` / ``y_pred`` [V, B, H, W], ``regions`` uint8 [V, B, W] -> (sums int64 [V, G, R, 5], maps int32
    [V, B, 2, G, W]); region codes >= n_regions are counted nowhere."""
    v, b, _, w = y_true.shape
    g = len(groups)
    sums = np.zeros((v, g, n_regions, 5), dtype=np.int64)
    maps = np.zeros((v, b, 2, g, w), dtype=np.int32)
    for i in range(v):
        for j in range(b):
            t = group_thickness(y_true[i, j], num_classes, groups)
            p = group_thickness(y_pred[i, j], num_classes, groups)
            maps[i, j, 0], maps[i, j, 1] = t, p
            r = regions[i, j].astype(np.int64)
            sel = r < n_regions
            d = t[:, sel] - p[:, sel]
            for gi in range(g):
                for s, val in enumerate((np.ones_like(d[gi]), t[gi, sel], p[gi, sel], np.abs(d[gi]), d[gi] * d[gi])):
                    np.add.at(sums[i, gi, :, s], r[sel], val)
    return sums, maps


def python_sums(y_true, y_pred, groups, regions, n_regions):
    """The same sums by a loop over every A-scan and pixel."""
    v, b, h, w = y_true.shape
    sums = [[[[0] * 5 for _ in range(n_regions)] for _ in groups] for _ in range(v)]
    for i in range(v):
        for j in range(b):
            for x in range(w):
                r = int(regions[i, j, x])
                if r >= n_regions:
                    continue
                for gi, (f, last) in enumerate(groups):
                    t = sum(1 for y in range(h) if f <= y_true[i, j, y, x] <= last)
                    p = sum(1 for y in range(h) if f <= y_pred[i, j, y, x] <= last)
                    acc = sums[i][gi][r]
                    acc[0] += 1
                    acc[1] += t
                    acc[2] += p
                    acc[3] += abs(t - p)
                    acc[4] += (t - p) ** 2
    return np.array(sums, dtype=np.int64)
