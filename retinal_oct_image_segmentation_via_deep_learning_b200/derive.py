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


def thickness_difference(thick_absdiff, width, spacing=None):
    """Biomarker_based_metrics.py:18-21 -- mean over the W columns of |thickness_t - thickness_p|; with a pixel
    ``spacing=(sy, sx)`` in the units of the row spacing: ``(sum / W) * sy``."""
    out = np.asarray(thick_absdiff, dtype=np.int64).astype(np.float64) / width
    return out if spacing is None else out * np.float64(spacing[0])


def boundary_errors(sum_sq, sum_abs, width, spacing=None):
    """MSE / RMSE / MAD of boundary-position rows (PixelError_based_metrics.py:14-17, 32-35;
    Contour_based_metrics.py:68-71 applied to integer boundary arrays of W columns).  With a pixel ``spacing=(sy, sx)``
    the positions are in the units of the row spacing: MSE ``(sum / W) * sy**2``, MAD ``(sum / W) * sy``."""
    mse = np.asarray(sum_sq, dtype=np.int64).astype(np.float64) / width
    mad = np.asarray(sum_abs, dtype=np.int64).astype(np.float64) / width
    if spacing is not None:
        sy = np.float64(spacing[0])
        mse, mad = mse * (sy * sy), mad * sy
    return {"boundary_mse": mse, "boundary_rmse": np.sqrt(mse), "boundary_mad": mad}


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
    contours (distance = sqrt(D2 / 4)), 1.0 for the voxel lattice of the 3-D surfaces.  Floating ``max_sq`` /
    ``p95_sq`` (physical squared distances of the 3-D surfaces with a spacing) are taken as they are."""
    n_pts = np.asarray(n_pts).astype(np.int64)
    max_sq = np.asarray(max_sq)
    max_sq = max_sq.astype(np.float64) if np.issubdtype(max_sq.dtype, np.floating) else max_sq.astype(np.int64)
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


SURFACE_DICE_MAX_REACH = 16      # lattice rows and lattice columns the surface Dice kernel reaches


def spacing_2d(spacing):
    """A B-scan pixel spacing ``(sy, sx)`` (rows = axial, columns = lateral; e.g. ``datasets.mhd_spacing(hdr)[-2:]``) ->
    tuple of 2 floats, or None for None.  ValueError unless both are finite and > 0 with squares that are normal doubles
    (the kernels work with ``wy = sy * sy`` and ``wx = sx * sx``)."""
    if spacing is None:
        return None
    try:
        sp = tuple(float(v) for v in np.asarray(spacing, dtype=np.float64).reshape(-1))
    except (TypeError, ValueError):
        raise ValueError(f"spacing must be 2 numbers (rows, columns), got {spacing!r}") from None
    if len(sp) != 2 or not all(np.isfinite(v) and v > 0 for v in sp):
        raise ValueError(f"spacing must be 2 finite numbers > 0 (rows, columns), got {spacing!r}")
    if not all(np.isfinite(v * v) and v * v >= np.finfo(np.float64).tiny for v in sp):
        raise ValueError(f"spacing {spacing!r}: the square of each entry must be a normal double")
    return sp


def surface_dice_spacing_limit(spacing):
    """The largest tolerance ``surface_dice`` accepts at pixel spacing ``(sy, sx)``: the kernel reaches 16 lattice rows and
    16 lattice columns, so tau must stay below ``sqrt(fl(w * 17**2) / 4.0)`` for ``w = sy**2`` and ``w = sx**2``."""
    sy, sx = spacing_2d(spacing)
    out = SURFACE_DICE_MAX_REACH + 1
    limit = min(np.sqrt(sy * sy * (out * out) / 4.0), np.sqrt(sx * sx * (out * out) / 4.0))
    return float(np.nextafter(limit, 0.0))


def surface_dice_spacing_tolerances(tolerances, spacing):
    """``surface_dice_tolerances`` with a pixel spacing: 1 to 4 finite tolerances ``>= 0`` in the units of the spacing, each
    at most ``surface_dice_spacing_limit(spacing)`` (ValueError naming that limit otherwise)."""
    taus = (tolerances,) if np.ndim(tolerances) == 0 else tuple(tolerances)
    if not 1 <= len(taus) <= SURFACE_DICE_MAX_TOL:
        raise ValueError(f"surface_dice takes 1 to {SURFACE_DICE_MAX_TOL} tolerances, got {len(taus)}")
    limit = surface_dice_spacing_limit(spacing)
    out = []
    for t in taus:
        try:
            v = float(t)
        except (TypeError, ValueError):
            raise ValueError(f"surface_dice tolerance {t!r} is not a number") from None
        if not 0.0 <= v < np.inf:
            raise ValueError(f"surface_dice tolerance {v} must be finite and >= 0")
        if v > limit:
            raise ValueError(f"surface_dice tolerance {v} reaches beyond {SURFACE_DICE_MAX_REACH} lattice rows or columns "
                             f"at spacing {tuple(spacing)}: the largest tolerance allowed is {limit!r}")
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


# ETDRS grid: region codes of ``etdrs_regions`` in this order.  The names are en-face index directions (b: B-scan index,
# x: column), not anatomy: which one is superior, inferior, nasal or temporal depends on the eye and on the device's
# B-scan order (INTEGRATION.md).
ETDRS_SECTORS = ("center", "inner_b-", "inner_x+", "inner_b+", "inner_x-", "outer_b-", "outer_x+", "outer_b+", "outer_x-")
ETDRS_RADII = (0.5, 1.5, 3.0)        # mm: 1, 3 and 6 mm diameters
NO_REGION = 255
SECTOR_STATS = ("n_ascans", "sum_true", "sum_pred", "sum_absdiff", "sum_sqdiff")     # last axis of the kernel's sums


def spacing_3d(spacing):
    """A volume spacing ``(sb, sy, sx)`` (B-scans, rows = axial, columns = lateral; ``datasets.mhd_spacing(hdr)``) ->
    tuple of 3 floats; ValueError unless all are finite and > 0."""
    try:
        sp = tuple(float(v) for v in np.asarray(spacing, dtype=np.float64).reshape(-1))
    except (TypeError, ValueError):
        raise ValueError(f"spacing must be 3 numbers (B-scans, rows, columns), got {spacing!r}") from None
    if len(sp) != 3 or not all(np.isfinite(v) and v > 0 for v in sp):
        raise ValueError(f"spacing must be 3 finite numbers > 0 (B-scans, rows, columns), got {spacing!r}")
    return sp


def etdrs_radii(radii):
    """``(R0, R1, R2)`` -> tuple of 3 floats; ValueError unless finite with ``0 < R0 <= R1 <= R2``."""
    try:
        r = tuple(float(v) for v in np.asarray(radii, dtype=np.float64).reshape(-1))
    except (TypeError, ValueError):
        raise ValueError(f"radii must be 3 numbers, got {radii!r}") from None
    if len(r) != 3 or not all(np.isfinite(v) for v in r) or not 0 < r[0] <= r[1] <= r[2]:
        raise ValueError(f"radii must be 3 finite numbers with 0 < R0 <= R1 <= R2, got {radii!r}")
    return r


def etdrs_regions(n_bscans, width, spacing, center, radii=ETDRS_RADII):
    """uint8 ``[n_bscans, width]`` ETDRS region of every A-scan (b, x) of one volume.

    With ``spacing = (sb, sy, sx)`` and ``center = (cb, cx)`` (fractional B-scan and column indices) the en-face position
    is ``pb = (b - cb) * sb``, ``px = (x - cx) * sx`` and ``r2 = pb * pb + px * px`` in float64.  With
    ``radii = (R0, R1, R2)``: region 0 (center) if ``r2 <= R0 * R0``, the inner ring if ``r2 <= R1 * R1``, the outer ring
    if ``r2 <= R2 * R2``, ``NO_REGION`` (255) otherwise.  A ring's quadrant is on the b side when ``|pb| > |px|`` and
    on the x side otherwise (diagonal ties go to x); regions 1-4 are inner b-, x+, b+, x-, regions 5-8 outer ones in the
    same order (``ETDRS_SECTORS``)."""
    sb, _, sx = spacing_3d(spacing)
    r0, r1, r2_ = etdrs_radii(radii)
    cb, cx = (float(v) for v in np.asarray(center, dtype=np.float64).reshape(2))
    if not (np.isfinite(cb) and np.isfinite(cx)):
        raise ValueError(f"center must be finite, got {center!r}")
    pb = (np.arange(int(n_bscans), dtype=np.float64) - cb)[:, None] * sb
    px = (np.arange(int(width), dtype=np.float64) - cx)[None, :] * sx
    r2 = pb * pb + px * px
    bside = np.abs(pb) > np.abs(px)
    quad = np.where(bside, np.where(pb < 0, 0, 2), np.where(px > 0, 1, 3))
    out = np.full(r2.shape, NO_REGION, dtype=np.uint8)
    out[r2 <= r2_ * r2_] = 5 + quad[r2 <= r2_ * r2_]
    out[r2 <= r1 * r1] = 1 + quad[r2 <= r1 * r1]
    out[r2 <= r0 * r0] = 0
    return out


def sector_thickness(sums, spacing):
    """Per-volume sector thickness from the exact sums of ``octm_sector_thickness_i32``: ``sums [V, G, R, 5]``
    (``SECTOR_STATS``) and the volume ``spacing = (sb, sy, sx)`` -> dict of float64 ``[V, G, R]`` arrays, NaN where a
    region holds no A-scan, plus ``n_ascans`` (int64).  In the units of the spacing, with n A-scans:

    - ``thickness_true`` = (sum t / n) * sy, ``thickness_pred`` = (sum p / n) * sy;
    - ``thickness_bias`` = ((sum p - sum t) / n) * sy;
    - ``thickness_mae`` = (sum |t - p| / n) * sy;
    - ``thickness_rmse`` = sqrt(sum (t - p)^2 / n) * sy;
    - ``volume_true`` = sum t * ((sb * sy) * sx), ``volume_pred`` likewise.
    """
    sb, sy, sx = spacing_3d(spacing)
    s = np.asarray(sums).astype(np.int64)
    n = s[..., 0]
    nf = np.where(n > 0, n, 1).astype(np.float64)
    nan = np.full(n.shape, np.nan)
    vox = (sb * sy) * sx

    def per(v):
        return np.where(n > 0, v, nan)
    return {"thickness_true": per(s[..., 1] / nf * sy), "thickness_pred": per(s[..., 2] / nf * sy),
            "thickness_bias": per((s[..., 2] - s[..., 1]) / nf * sy), "thickness_mae": per(s[..., 3] / nf * sy),
            "thickness_rmse": per(np.sqrt(s[..., 4] / nf) * sy),
            "volume_true": per(s[..., 1] * vox), "volume_pred": per(s[..., 2] * vox), "n_ascans": n}


SECTOR_SUMMARY = ("abs_bias", "bias", "mae", "rmse", "thickness_true", "thickness_pred")


def sector_thickness_summary(per_volume):
    """Dataset-level sector thickness from ``sector_thickness`` output: per (group, sector) the mean over the volumes
    whose region holds at least one A-scan, summed in volume order, of |bias|, bias, MAE, RMSE, true and predicted
    thickness (``SECTOR_SUMMARY`` order), float64 ``[G, R]`` each (NaN where no volume covers the region), and
    ``n_volumes`` (int64 ``[G, R]``), the number of volumes covering it."""
    src = {"abs_bias": np.abs(per_volume["thickness_bias"]), "bias": per_volume["thickness_bias"],
           "mae": per_volume["thickness_mae"], "rmse": per_volume["thickness_rmse"],
           "thickness_true": per_volume["thickness_true"], "thickness_pred": per_volume["thickness_pred"]}
    covered = np.asarray(per_volume["n_ascans"]) > 0
    cnt = covered.sum(axis=0).astype(np.int64)
    out = {}
    for name in SECTOR_SUMMARY:
        v = np.asarray(src[name], dtype=np.float64)
        acc = np.zeros(v.shape[1:])
        for i in range(v.shape[0]):
            acc = acc + np.where(covered[i], v[i], 0.0)
        with np.errstate(invalid="ignore", divide="ignore"):
            out[name] = np.where(cnt > 0, acc / np.maximum(cnt, 1), np.nan)
    out["n_volumes"] = cnt
    return out


SECTOR_MAX_GROUPS = 16


def sector_groups(classes, num_classes):
    """``classes`` of ``suite.sector_thickness`` -> tuple of ``(first, last)`` class pairs: None gives one group per class;
    otherwise 1 to 16 entries, each a class or a ``(first, last)`` pair with ``0 <= first <= last <= num_classes - 1``."""
    k = int(num_classes)
    if classes is None:
        entries = list(range(k))
    else:
        entries = list(classes)
    if not 1 <= len(entries) <= SECTOR_MAX_GROUPS:
        raise ValueError(f"classes: 1 to {SECTOR_MAX_GROUPS} groups, got {len(entries)}")
    out = []
    for e in entries:
        pair = (e, e) if np.ndim(e) == 0 else tuple(e)
        if len(pair) != 2 or not all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in pair):
            raise ValueError(f"classes: each entry must be a class or a (first, last) pair of ints, got {e!r}")
        f, last = int(pair[0]), int(pair[1])
        if not 0 <= f <= last <= k - 1:
            raise ValueError(f"classes: group {e!r} needs 0 <= first <= last <= {k - 1}")
        out.append((f, last))
    return tuple(out)


def sector_centers(center, n_volumes, n_bscans, width):
    """``center`` of ``suite.sector_thickness`` -> float64 ``[V, 2]`` (B-scan, column) fractional indices: None gives the
    geometric centre ``((B - 1) / 2, (W - 1) / 2)`` of every volume, one pair is used for every volume, and a ``[V, 2]``
    array gives one per volume.  ValueError for another shape or a value that is not finite."""
    if center is None:
        return np.tile(np.array([(n_bscans - 1) / 2.0, (width - 1) / 2.0]), (n_volumes, 1))
    try:
        c = np.asarray(center, dtype=np.float64)
    except (TypeError, ValueError):
        raise ValueError(f"center must be a (b, x) pair or a [V, 2] array, got {center!r}") from None
    if c.shape == (2,):
        c = np.tile(c, (n_volumes, 1))
    if c.shape != (n_volumes, 2):
        raise ValueError(f"center must be a (b, x) pair or a [{n_volumes}, 2] array, got shape {c.shape}")
    if not np.all(np.isfinite(c)):
        raise ValueError("center must be finite")
    return c
