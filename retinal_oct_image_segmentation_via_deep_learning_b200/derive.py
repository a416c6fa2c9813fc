"""Float64 epilogue: the reference's scalar expressions evaluated from the GPU's exact integers.

Every formula keeps the operation order of the reference line it cites (paths relative to the
reference's ``Metrics/``), so the results are bit-identical to running the reference per class on
``(gt == c, pr == c)`` int64 masks (SURVEY.md 8a; pinned by tests/test_derive.py against the
golden vectors produced by the executed reference).  Inputs are numpy integer arrays of any shape
(typically ``[N, K]``); outputs are float64 arrays of the same shape.
"""
from __future__ import annotations

import numpy as np

EPS = 1e-7   # denominator guard used throughout the reference (e.g. Region_based_metrics.py:15)


def class_counts(confusion):
    """``[..., K, K]`` confusion matrices ``cm[t][p]`` -> per-class int64 TP, FP, FN, TN, N."""
    cm = np.asarray(confusion).astype(np.int64)
    tp = np.diagonal(cm, axis1=-2, axis2=-1)
    fn = cm.sum(axis=-1) - tp            # true class c, predicted something else
    fp = cm.sum(axis=-2) - tp            # predicted class c, truth something else
    n = cm.sum(axis=(-2, -1))[..., None] + np.zeros_like(tp)
    tn = n - tp - fn - fp
    return tp, fp, fn, tn, n


def count_metrics(tp, fp, fn, tn, n):
    """The twelve count-derived scalars of the reference, per class."""
    tp, fp, fn, tn, n = (np.asarray(v, dtype=np.int64) for v in (tp, fp, fn, tn, n))
    sum_t, sum_p = tp + fn, tp + fp
    with np.errstate(divide="ignore", invalid="ignore"):
        err = (fp + fn).astype(np.float64) / n      # mean of a 0/1 array == exact count / size
        return {
            # ConfusionMatrix_based_metrics.py:14-17  (TP + TN) / prod(shape), no epsilon
            "accuracy": (tp + tn) / n,
            # :30-32  TP / (TP + FN + 1e-7)
            "sensitivity": tp / (tp + fn + EPS),
            # :45-47  TP / (TP + FP + 1e-7)
            "cm_precision": tp / (tp + fp + EPS),
            # :60-62  TN / (TN + FP + 1e-7)
            "specificity": tn / (tn + fp + EPS),
            # Region_based_metrics.py:13-15  2.*I / (sum(t) + sum(p) + 1e-7)
            "dice_coefficient": (2.0 * tp) / (sum_t + sum_p + EPS),
            # :28-30  I / (sum(t) + sum(p) - I + 1e-7)
            "iou_score": tp / (sum_t + sum_p - tp + EPS),
            # :43-45  I / (sum(p) + 1e-7)
            "region_precision": tp / (sum_p + EPS),
            # :58-60  I / (sum(t) + 1e-7)
            "recall": tp / (sum_t + EPS),
            # PixelError_based_metrics.py:14-17, 32-35 and Contour_based_metrics.py:68-71 on 0/1 masks
            "mean_squared_error": err,
            "root_mean_squared_error": np.sqrt(err),
            "mad": err,
            # Biomarker_based_metrics.py:34-38  |sum(t)/size - sum(p)/size|
            "vascularity_index": np.abs(sum_t / n - sum_p / n),
        }


def thickness_difference(thick_absdiff, width):
    """Biomarker_based_metrics.py:18-21 -- mean over the W columns of |thickness_t - thickness_p|."""
    return np.asarray(thick_absdiff, dtype=np.int64).astype(np.float64) / width


def boundary_errors(sum_sq, sum_abs, width):
    """MSE / RMSE / MAD of boundary-position rows (PixelError_based_metrics.py:14-17, 32-35;
    Contour_based_metrics.py:68-71 applied to integer boundary arrays of W columns)."""
    mse = np.asarray(sum_sq, dtype=np.int64).astype(np.float64) / width
    return {"boundary_mse": mse, "boundary_rmse": np.sqrt(mse),
            "boundary_mad": np.asarray(sum_abs, dtype=np.int64).astype(np.float64) / width}


def _lerp(a, b, t):
    """numpy's ``_lerp`` (lib/_function_base_impl.py) for the linear percentile."""
    d = b - a
    out = a + d * t
    alt = b - d * (1 - t)
    return np.where(t >= 0.5, alt, out)


def contour_metrics(n_pts, max_sq, p95_sq, sum_dist, lattice=4.0):
    """hausdorff / hd95 / assd from the contour kernel's integers (Contour_based_metrics.py:22, 39, 56).

    ``n_pts [..., 2]`` (true, pred); ``max_sq [..., 2]``, ``p95_sq [..., 2, 2]``, ``sum_dist [..., 2]``
    indexed by direction (0: pred vertices -> true contour = ``d1``; 1: true -> pred = ``d2``).
    Entries whose masks have no contour (the reference raises IndexError) come back as NaN.
    ``lattice``: squared length unit of the integer distances -- 4.0 for the doubled lattice of the 2-D
    contours (distance = sqrt(D2 / 4)), 1.0 for the voxel lattice of the 3-D surfaces."""
    n_pts = np.asarray(n_pts).astype(np.int64)
    max_sq = np.asarray(max_sq).astype(np.int64)
    p95 = np.asarray(p95_sq).astype(np.float64)
    valid = (n_pts[..., 0] > 0) & (n_pts[..., 1] > 0)
    m = np.stack([n_pts[..., 1], n_pts[..., 0]], axis=-1)         # query count per direction
    msafe = np.maximum(m, 1)
    hd = np.sqrt(np.maximum(max_sq[..., 0], max_sq[..., 1]).astype(np.float64) / lattice)
    # numpy percentile, method "linear": virtual index (m - 1) * 0.95
    pos = (msafe - 1) * (95 / 100)
    gamma = pos - np.floor(pos)
    lo = np.sqrt(p95[..., 0] / lattice)
    hi = np.sqrt(p95[..., 1] / lattice)
    pct = _lerp(lo, hi, gamma)
    hd95 = np.maximum(pct[..., 0], pct[..., 1])
    mean = np.asarray(sum_dist, dtype=np.float64) / msafe
    assd = (mean[..., 0] + mean[..., 1]) / 2
    nan = np.full(valid.shape, np.nan)
    return {"hausdorff_distance": np.where(valid, hd, nan),
            "hausdorff_distance_95": np.where(valid, hd95, nan),
            "assd": np.where(valid, assd, nan),
            "contour_valid": valid}


SURFACE_DICE_MAX_TOL = 4         # OCTM_SURFACE_DICE_MAX_TOL: tolerances per call
SURFACE_DICE_MAX_TAU = 8.0       # pixels; T(8) = OCTM_SURFACE_DICE_MAX_SQ = 256


def surface_dice_threshold(tau):
    """Integer threshold of tolerance ``tau`` (pixels): the largest squared doubled-lattice distance D with
    ``sqrt(D / 4.0) <= tau``, tested with the expression every contour distance of the suite is reported through, so
    that "within tau" means what a user computes from those distances, boundary cases included."""
    t = float(tau)
    d = int(np.floor(4.0 * t * t))
    while d > 0 and not np.sqrt(d / 4.0) <= t:
        d -= 1
    while np.sqrt((d + 1) / 4.0) <= t:
        d += 1
    return d


def surface_dice_tolerances(tolerances):
    """A tolerance or a sequence of 1 to 4 of them -> tuple of floats; ValueError outside ``0 <= tau <= 8`` (NaN
    included) or for an empty or longer list."""
    taus = (tolerances,) if np.ndim(tolerances) == 0 else tuple(tolerances)
    if not 1 <= len(taus) <= SURFACE_DICE_MAX_TOL:
        raise ValueError(f"surface_dice takes 1 to {SURFACE_DICE_MAX_TOL} tolerances, got {len(taus)}")
    out = []
    for t in taus:
        try:
            v = float(t)
        except (TypeError, ValueError):
            raise ValueError(f"surface_dice tolerance {t!r} is not a number") from None
        if not 0.0 <= v <= SURFACE_DICE_MAX_TAU:          # False for NaN
            raise ValueError(f"surface_dice tolerance {v} outside [0, {SURFACE_DICE_MAX_TAU}] pixels")
        out.append(v)
    return tuple(out)


def surface_dice(n_surf, n_within):
    """Normalized surface Dice per tolerance from the exact counts of ``octm_surface_dice_u8``: ``n_surf [..., 2]``
    (|V_t|, |V_p|) and ``n_within [..., 2, T]`` -> float64 ``[..., T]`` = (n_within[..., 0, :] + n_within[..., 1, :]) /
    (|V_t| + |V_p|).  NaN when both boundaries are empty (class absent from or filling both maps), 0 when exactly one
    is (as MONAI)."""
    ns = np.asarray(n_surf).astype(np.int64)
    nw = np.asarray(n_within).astype(np.int64)
    tot = (ns[..., 0] + ns[..., 1])[..., None]
    num = (nw[..., 0, :] + nw[..., 1, :]).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(tot > 0, num / np.maximum(tot, 1), np.nan)


COMPONENT_METRICS = ("component_count_error", "component_recall", "component_precision", "component_f1")


def component_metrics(n_comp, n_hit):
    """Lesion-wise detection scores from the exact counts of ``octm_components_u8``: ``n_comp [..., 2]`` (components of
    y_true, y_pred) and ``n_hit [..., 2]`` (of those, the ones that share a pixel with the other map's class) -> float64
    ``[...]`` arrays keyed by ``COMPONENT_METRICS``:

    - ``component_count_error`` = |n_t - n_p|;
    - ``component_recall`` = hit_t / n_t, NaN when n_t == 0;
    - ``component_precision`` = hit_p / n_p, NaN when n_p == 0;
    - ``component_f1`` = 2 P R / (P + R): NaN when n_t == n_p == 0, 0 when exactly one of them is 0 or P + R == 0.
    """
    nc = np.asarray(n_comp).astype(np.int64)
    nh = np.asarray(n_hit).astype(np.int64)
    nt, npred = nc[..., 0], nc[..., 1]
    with np.errstate(divide="ignore", invalid="ignore"):
        rec = np.where(nt > 0, nh[..., 0] / np.maximum(nt, 1), np.nan)
        prec = np.where(npred > 0, nh[..., 1] / np.maximum(npred, 1), np.nan)
        both = (nt > 0) & (npred > 0)
        r0, p0 = np.where(both, rec, 0.0), np.where(both, prec, 0.0)
        s = r0 + p0
        f1 = np.where(s > 0, 2.0 * p0 * r0 / np.where(s > 0, s, 1.0), 0.0)
    f1 = np.where((nt == 0) & (npred == 0), np.nan, f1)
    return {"component_count_error": np.abs(nt - npred).astype(np.float64), "component_recall": rec,
            "component_precision": prec, "component_f1": f1}
