"""Batched, device-resident entry points of the metric suite (the host side of the C ABI).

``y_true`` / ``y_pred`` are CUDA ``torch.uint8`` label maps ``[N, H, W]`` with values ``< num_classes``.
torch is used only for device memory and streams; all arithmetic on label data happens in the
hand-written kernels of ``liboctm.so`` (no CPU or torch fallback), and the float64 ratios are
evaluated on the host from the kernels' exact integers (``derive.py``).

    res = evaluate(y_true, y_pred, num_classes=8)        # one fused label pass + contour kernels
    res.metrics()["dice_coefficient"]                      # float64 [N, K], reference operation order
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib, derive

DEFAULT_MAX_PTS = 2048       # contour vertices kept per (item, class, map) on the first attempt (at least; see default_max_pts)
MAX_MAX_PTS = 1 << 16        # bound of the retry for items whose contour overflowed max_pts (8 B of scratch per vertex)


def default_max_pts(width):
    """First-attempt vertex bound: a layer boundary crossing a W-pixel image has 2 W + sum |dh| vertices (2.7 W on the
    synthetic layers), so the bound grows with the width -- 2048 up to W = 512, 4 W beyond (a 1024-wide HC-MS B-scan would
    otherwise overflow on every contour and be redone)."""
    return max(DEFAULT_MAX_PTS, min(MAX_MAX_PTS, 4 * int(width)))


def default_max_pts_all(width):
    """First-attempt vertex bound of ``mode="all"``: a layer band has two boundaries (its upper and its lower one, each
    about 2.7 W vertices on the synthetic layers), hence 8 W."""
    return max(DEFAULT_MAX_PTS, 8 * int(width))


def crack_bound(height, width):
    """Largest possible all-contour vertex count of one class: every crack between 4-adjacent pixels."""
    return (int(height) - 1) * int(width) + int(height) * (int(width) - 1)


CONTOUR_MODES = ("first", "all")
CONTOUR_CHUNK_BYTES = 4 << 30   # vertex + squared-distance scratch per chunk of items (grow-only, reused)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_pair(y_true, y_pred):
    for name, t in (("y_true", y_true), ("y_pred", y_pred)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise TypeError(f"{name} must be a CUDA torch tensor (got {type(t).__name__}); "
                            "use the Metrics/ drop-in functions for host arrays")
        if t.dtype not in (torch.uint8, torch.bool):
            raise TypeError(f"{name} must be uint8 (or bool), got {t.dtype}")
    if y_true.shape != y_pred.shape:
        raise ValueError(f"shape mismatch: {tuple(y_true.shape)} vs {tuple(y_pred.shape)}")
    if y_true.device != y_pred.device:
        raise ValueError("y_true and y_pred are on different devices")
    if y_true.dim() == 2:
        y_true, y_pred = y_true[None], y_pred[None]
    if y_true.dim() != 3:
        raise ValueError("expected [N, H, W] or [H, W] label maps")
    cast = lambda t: (t.view(torch.uint8) if t.dtype == torch.bool else t).contiguous()   # noqa: E731
    return cast(y_true), cast(y_pred)


@dataclass
class LabelPassOut:
    """Exact integers of the fused label pass (device tensors; u64/u32 stored as int64/int32 bits)."""
    num_classes: int
    height: int
    width: int
    counts: torch.Tensor | None = None          # [N, K, K]   cm[t][p]
    thick_absdiff: torch.Tensor | None = None   # [N, K]
    bnd_sq: torch.Tensor | None = None          # [N, K-1]
    bnd_abs: torch.Tensor | None = None         # [N, K-1]
    bnd_true: torch.Tensor | None = None        # [N, K-1, W] int32
    bnd_pred: torch.Tensor | None = None
    first_pos: torch.Tensor | None = None       # [N, 2, K]  uint32 bits
    unsorted: torch.Tensor | None = None        # [N] bit 0 / 1: a column of y_true / y_pred is not in class order


class _Timed:
    """Bracket a launch with CUDA events on the current stream when a timers dict is supplied."""

    def __init__(self, timers, key):
        self.timers, self.key = timers, key

    def __enter__(self):
        if self.timers is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.timers is not None:
            self.b.record()
            self.timers.setdefault(self.key, []).append((self.a, self.b))


def label_pass(y_true, y_pred, num_classes, *, counts=True, columns=True, seeds=False, boundaries=False,
               timers=None, certify=False):
    """One read of both label tensors -> confusion matrices, column-scan sums, contour seeds; ``certify`` adds the
    per-item layering certificate ``unsorted`` (needs counts, columns and seeds)."""
    yt, yp = _check_pair(y_true, y_pred)
    n, h, w = yt.shape
    k = int(num_classes)
    dev = yt.device
    out = LabelPassOut(k, h, w)
    with torch.cuda.device(dev):
        if counts:
            out.counts = torch.empty((n, k, k), dtype=torch.int64, device=dev)
        if columns or boundaries:
            out.thick_absdiff = torch.empty((n, k), dtype=torch.int64, device=dev)
            out.bnd_sq = torch.empty((n, k - 1), dtype=torch.int64, device=dev)
            out.bnd_abs = torch.empty((n, k - 1), dtype=torch.int64, device=dev)
        if boundaries:
            out.bnd_true = torch.empty((n, k - 1, w), dtype=torch.int32, device=dev)
            out.bnd_pred = torch.empty((n, k - 1, w), dtype=torch.int32, device=dev)
        if seeds:
            out.first_pos = torch.empty((n, 2, k), dtype=torch.int32, device=dev)
        if certify:
            out.unsorted = torch.empty((n,), dtype=torch.int32, device=dev)
        with _Timed(timers, "label_pass"):
            _lib.call("octm_label_pass_sorted_u8", _ptr(yt), _ptr(yp), n, h, w, k, _ptr(out.counts),
                      _ptr(out.thick_absdiff), _ptr(out.bnd_sq), _ptr(out.bnd_abs), _ptr(out.bnd_true),
                      _ptr(out.bnd_pred), _ptr(out.first_pos), _ptr(out.unsorted), _stream())
    return out


def confusion(y_true, y_pred, num_classes):
    """K1 alone: ``int64 [N, K, K]`` confusion matrices (items may have any trailing shape)."""
    for t in (y_true, y_pred):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype not in (torch.uint8, torch.bool):
            raise TypeError("confusion() takes CUDA uint8/bool tensors")
    if y_true.shape != y_pred.shape:
        raise ValueError("shape mismatch")
    yt = (y_true.view(torch.uint8) if y_true.dtype == torch.bool else y_true).contiguous()
    yp = (y_pred.view(torch.uint8) if y_pred.dtype == torch.bool else y_pred).contiguous()
    n = yt.shape[0]
    elems = yt[0].numel() if n else 1
    k = int(num_classes)
    out = torch.empty((n, k, k), dtype=torch.int64, device=yt.device)
    with torch.cuda.device(yt.device):
        _lib.call("octm_confusion_u8", _ptr(yt), _ptr(yp), n, elems, k, _ptr(out), _stream())
    return out


_FLOAT_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16,
                 torch.float64: _lib.DTYPE_F64}


def boundary_error(bnd_true, bnd_pred):
    """K3 alone on caller-supplied boundary positions ``[N, Kb, W]`` -> ``(sum_sq, sum_abs)`` per ``[N, Kb]`` row.

    Integer positions (e.g. ``b_k(x)`` extracted from label maps) give exact int64 sums; floating
    positions (the soft-argmax rows a layer model such as SD-LayerNet's ``LayerEngine`` produces) give
    float64 sums accumulated in a fixed order."""
    if bnd_true.shape != bnd_pred.shape or bnd_true.dim() != 3:
        raise ValueError("expected two [N, Kb, W] tensors of equal shape")
    n, kb, w = bnd_true.shape
    if bnd_true.is_floating_point() or bnd_pred.is_floating_point():
        dt = torch.promote_types(bnd_true.dtype, bnd_pred.dtype)
        bt, bp = bnd_true.to(dt).contiguous(), bnd_pred.to(dt).contiguous()
        sq = torch.empty((n, kb), dtype=torch.float64, device=bt.device)
        ab = torch.empty((n, kb), dtype=torch.float64, device=bt.device)
        with torch.cuda.device(bt.device):
            _lib.call("octm_boundary_error_float", _ptr(bt), _ptr(bp), _FLOAT_DTYPES[dt], n, kb, w, _ptr(sq), _ptr(ab),
                      _stream())
        return sq, ab
    bt, bp = bnd_true.to(torch.int32).contiguous(), bnd_pred.to(torch.int32).contiguous()
    sq = torch.empty((n, kb), dtype=torch.int64, device=bt.device)
    ab = torch.empty((n, kb), dtype=torch.int64, device=bt.device)
    with torch.cuda.device(bt.device):
        _lib.call("octm_boundary_error_i32", _ptr(bt), _ptr(bp), n, kb, w, _ptr(sq), _ptr(ab), _stream())
    return sq, ab


def labels_from_boundaries(boundaries, height):
    """Boundary rows ``[N, Kb, W]`` (int or float, CUDA) -> uint8 label maps ``[N, height, W]``:
    ``label[i, y, x] = #{k : b_k(i, x) <= y}``.  The inverse of the label pass's boundary rows on layered maps;
    this is how boundary-curve annotations (Duke ``manualLayers``, HC-MS control points, the soft rows of a layer
    model) become inputs of the mask metrics.  Rows may be unsorted, out of range or NaN (= boundary absent)."""
    if not isinstance(boundaries, torch.Tensor) or not boundaries.is_cuda or boundaries.dim() != 3:
        raise TypeError("expected a CUDA tensor [N, Kb, W]")
    n, kb, w = boundaries.shape
    if kb > 15:
        raise ValueError("at most 15 boundaries (16 classes)")
    if boundaries.is_floating_point():
        b, dt = boundaries.to(torch.float32).contiguous(), _lib.DTYPE_F32
    else:
        b, dt = boundaries.to(torch.int32).contiguous(), _lib.DTYPE_I32
    out = torch.empty((n, int(height), w), dtype=torch.uint8, device=b.device)
    with torch.cuda.device(b.device):
        _lib.call("octm_labels_from_boundaries", _ptr(b), dt, n, kb, int(height), w, _ptr(out), _stream())
    return out


def boundary_metrics(bnd_true, bnd_pred):
    """``mean_squared_error`` / ``root_mean_squared_error`` / ``mad`` of the reference applied to every
    boundary row: dict of float64 ``[N, Kb]`` CUDA tensors (reference: PixelError_based_metrics.py:14-35,
    Contour_based_metrics.py:68-71)."""
    sq, ab = boundary_error(bnd_true, bnd_pred)
    w = bnd_true.shape[-1]
    mse = sq.to(torch.float64) / w
    return {"boundary_mse": mse, "boundary_rmse": torch.sqrt(mse), "boundary_mad": ab.to(torch.float64) / w}


def topology_violations(positions):
    """``relu(pos[:, :-1] - pos[:, 1:])`` of ``LayerEngine.get_topology_violations`` (SD_Layer_Net/layer_engine.py:74-76),
    reduced over the width: ``(sum_violation float64 [N, Kb-1], n_violations int32 [N, Kb-1])``."""
    if not isinstance(positions, torch.Tensor) or not positions.is_cuda or positions.dim() != 3:
        raise TypeError("positions must be a CUDA tensor [N, Kb, W]")
    pos = positions if positions.is_floating_point() else positions.to(torch.float64)
    pos = pos.contiguous()
    n, kb, w = pos.shape
    if kb < 2:
        raise ValueError("need at least two boundaries")
    sv = torch.empty((n, kb - 1), dtype=torch.float64, device=pos.device)
    nv = torch.empty((n, kb - 1), dtype=torch.int32, device=pos.device)
    with torch.cuda.device(pos.device):
        _lib.call("octm_topology_violations_float", _ptr(pos), _FLOAT_DTYPES[pos.dtype], n, kb, w, _ptr(sv), _ptr(nv), _stream())
    return sv, nv


@dataclass
class ContourOut:
    """Exact integers (and the float64 distance sums) of the contour kernels, device tensors."""
    n_pts: torch.Tensor        # [N, K, 2]   uint32 bits
    flags: torch.Tensor        # [N, K]
    max_sq: torch.Tensor       # [N, K, 2]
    p95_sq: torch.Tensor       # [N, K, 2, 2]
    sum_dist: torch.Tensor     # [N, K, 2]   float64
    verts: torch.Tensor | None = None     # [N, K, 2, max_pts] when requested
    sq: torch.Tensor | None = None        # [N, K, 2, max_pts] when requested
    max_pts: int = 0
    mode: str = "first"                   # "first": contour [0] only; "all": every contour of each class


_SCRATCH = {}      # (device, stream) -> grow-only int32 scratch for contour vertices (pure workspace, never returned)


_STAGING = {}      # device -> (copy stream, grow-only uint8 staging buffer of evaluate_host)


def _staging(dev, nbytes):
    """Copy stream and device staging buffer of ``evaluate_host``, cached per device: a fresh cudaMalloc of
    a few hundred MB per call costs more than the copies it serves."""
    ent = _STAGING.get(dev)
    if ent is None or ent[1].numel() < nbytes:
        stream = ent[0] if ent is not None else torch.cuda.Stream(device=dev)
        _STAGING.pop(dev, None)
        ent = (stream, torch.empty((nbytes,), dtype=torch.uint8, device=dev))
        _STAGING[dev] = ent
    return ent


def _vertex_scratch(dev, numel):
    """Grow-only int32 workspace, one per (device, stream): every consumer of a buffer is enqueued on the stream it
    is keyed by, so reuse is stream-ordered and two streams never share scratch."""
    key = (dev, torch.cuda.current_stream(dev).cuda_stream)
    buf = _SCRATCH.get(key)
    if buf is None or buf.numel() < numel:
        _SCRATCH.pop(key, None)
        buf = None
        buf = torch.empty((numel,), dtype=torch.int32, device=dev)
        _SCRATCH[key] = buf
    return buf[:numel]


def _contour_outputs(n, k, dev):
    """Empty ``n_pts``, ``flags``, ``max_sq``, ``p95_sq``, ``sum_dist`` of ``n`` items (the ``ContourOut`` order)."""
    i32 = dict(dtype=torch.int32, device=dev)
    return (torch.empty((n, k, 2), **i32), torch.empty((n, k), **i32), torch.empty((n, k, 2), **i32),
            torch.empty((n, k, 2, 2), **i32), torch.empty((n, k, 2), dtype=torch.float64, device=dev))


def _contour_chunk(yt, yp, k, max_pts, mode, want_verts, want_sq, timers=None, first_pos=None, bnd=None, unsorted=None):
    """One chunk of ``contour_pass``.  Metrics alone take the one-call entry point of ``mode`` on the shared scratch;
    requested vertices or squared distances take the vertex emitter of ``mode``, then ``octm_contour2d_distance``."""
    n, h, w = yt.shape
    dev = yt.device
    n_pts, flags, max_sq, p95, sums = _contour_outputs(n, k, dev)
    bt, bp = (None, None) if bnd is None else bnd
    if not want_verts and not want_sq:
        # stream-ordered reuse: every consumer of the scratch is enqueued on the same stream
        scratch = _vertex_scratch(dev, (int(_lib.load().octm_contour2d_workspace_bytes(n, h, w, k, max_pts)) + 3) // 4)
        with _Timed(timers, "contour"):
            if mode == "first":
                # layered pairs (with boundary rows and certificate) are measured from the rows, the rest from vertex lists
                _lib.call("octm_contour2d_metrics_u8", _ptr(yt), _ptr(yp), n, h, w, k, _ptr(first_pos), _ptr(bt), _ptr(bp),
                          _ptr(unsorted), max_pts, _ptr(n_pts), _ptr(flags), _ptr(max_sq), _ptr(p95), _ptr(sums),
                          _ptr(scratch), scratch.numel() * 4, _stream())
            else:
                _lib.call("octm_contour2d_all_u8", _ptr(yt), _ptr(yp), n, h, w, k, max_pts, _ptr(n_pts), _ptr(flags),
                          _ptr(max_sq), _ptr(p95), _ptr(sums), _ptr(scratch), scratch.numel() * 4, _stream())
        return ContourOut(n_pts, flags, max_sq, p95, sums, None, None, max_pts, mode)
    verts = torch.empty((n, k, 2, max_pts), dtype=torch.int32, device=dev)
    sq = torch.empty((n, k, 2, max_pts), dtype=torch.int32, device=dev)
    with _Timed(timers, "contour_trace"):
        if mode == "first":
            _lib.call("octm_contour2d_trace_u8", _ptr(yt), _ptr(yp), n, h, w, k, _ptr(first_pos), _ptr(bt), _ptr(bp),
                      max_pts, _ptr(verts), _ptr(n_pts), _ptr(flags), _stream())
        else:
            _lib.call("octm_contour2d_all_vertices_u8", _ptr(yt), _ptr(yp), n, h, w, k, max_pts, _ptr(verts),
                      _ptr(n_pts), _ptr(flags), _stream())
    with _Timed(timers, "contour_distance"):
        _lib.call("octm_contour2d_distance", _ptr(verts), _ptr(n_pts), n, k, max_pts, h, w, _ptr(max_sq), _ptr(p95),
                  _ptr(sums), _ptr(sq), 1 if want_sq else 0, _stream())
    return ContourOut(n_pts, flags, max_sq, p95, sums, verts if want_verts else None, sq if want_sq else None, max_pts,
                      mode)


def contour_pass(y_true, y_pred, num_classes, first_pos=None, *, max_pts=None, return_vertices=False,
                 return_sq=False, timers=None, check_overflow=True, boundaries=None, unsorted=None, mode="first"):
    """Contour ``[0]`` of every class mask of both maps, then hausdorff / hd95 / assd integers.

    ``mode="all"`` measures EVERY contour of each class instead (build-defined, no reference counterpart): the vertex
    set of a class is the midpoint of every crack between two 4-adjacent pixels exactly one of which is in the class,
    each once, in raster order of the doubled lattice (``octm_contour2d_all_vertices_u8``); ``n_pts`` is its exact
    size.  ``first_pos``, ``boundaries`` and ``unsorted`` are not used then, and the default bound is
    ``default_max_pts_all(W)``.

    ``boundaries``: optional ``(bnd_true, bnd_pred)`` int32 ``[N, K-1, W]`` of the label pass; with them the
    contours of layered maps are verified and emitted in parallel instead of walked (same vertices).
    ``unsorted``: optional layering certificate ``[N]`` of ``label_pass(certify=True)``; with it (and the boundary
    rows) certified items are verified and measured from the boundary rows alone.

    Items are processed in chunks so the vertex workspace stays under ~1 GiB; items whose contour is
    longer than ``max_pts`` are re-run on their own with a larger bound."""
    if mode not in CONTOUR_MODES:
        raise ValueError(f"mode must be one of {CONTOUR_MODES}, got {mode!r}")
    yt, yp = _check_pair(y_true, y_pred)
    n, h, w = yt.shape
    k = int(num_classes)
    if max_pts is None:
        max_pts = default_max_pts_all(w) if mode == "all" else default_max_pts(w)
    max_pts = (int(max_pts) + 3) & ~3
    if h < 2 or w < 2:
        raise ValueError("Input array must be at least 2x2.")     # skimage's message for find_contours
    dev = yt.device
    if mode == "all":
        first_pos = boundaries = unsorted = None
    with torch.cuda.device(dev):
        if first_pos is None and mode == "first":
            first_pos = torch.empty((n, 2, k), dtype=torch.int32, device=dev)
            tmp = torch.empty((n, k), dtype=torch.int32, device=dev)
            for m, src in enumerate((yt, yp)):
                _lib.call("octm_first_pos_u8", _ptr(src), n, h * w, k, _ptr(tmp), _stream())
                first_pos[:, m, :] = tmp
        keep = return_vertices or return_sq
        if n == 0:
            return ContourOut(*_contour_outputs(0, k, dev), None, None, max_pts, mode)
        per_item = k * 2 * max_pts * 4 * 2          # vertices + squared-distance scratch
        chunk = n if keep else max(1, min(n, CONTOUR_CHUNK_BYTES // per_item))
        parts = []
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            parts.append(_contour_chunk(yt[s:e], yp[s:e], k, max_pts, mode, return_vertices, return_sq, timers,
                                        None if first_pos is None else first_pos[s:e],
                                        None if boundaries is None else (boundaries[0][s:e], boundaries[1][s:e]),
                                        None if unsorted is None else unsorted[s:e]))
        if len(parts) == 1:
            out = parts[0]
        else:
            cat = lambda f: torch.cat([getattr(p, f) for p in parts])      # noqa: E731
            out = ContourOut(cat("n_pts"), cat("flags"), cat("max_sq"), cat("p95_sq"), cat("sum_dist"), None, None,
                             max_pts, mode)
        if check_overflow:
            _retry_overflow(out, yt, yp, k, first_pos, keep)
    return out


def _retry_overflow(out, yt, yp, k, first_pos, keep=False):
    """Re-run, with a larger vertex bound, the (rare) items whose contour overflowed ``max_pts``.  The bound
    escalates geometrically (x8 per round, up to MAX_MAX_PTS) and every round is chunked so that its vertex and
    distance scratch stays below CONTOUR_CHUNK_BYTES, like the first pass.  Returns True when something was
    redone.  Costs one device->host sync per round.

    ``mode="all"`` counts every vertex even past the bound, so a single round redoes the overflowed items with the
    largest count (rounded up to a multiple of 4) as the bound; no count exceeds ``crack_bound(H, W)``."""
    over_bits = _lib.CF_TRUE_OVERFLOW | _lib.CF_PRED_OVERFLOW
    over = ((out.flags & over_bits) != 0).any(dim=1)
    if not bool(over.any()):
        return False
    idx = torch.nonzero(over).flatten()
    big = max(int(out.max_pts), 8)
    while idx.numel():
        if out.mode == "all":
            big = (int(out.n_pts[idx].max()) + 3) & ~3
            if keep:
                raise _lib.OctmError(f"a class has {big} boundary vertices (rounded up to a multiple of 4), more than "
                                     f"max_pts={out.max_pts}; pass max_pts >= {big}")
        else:
            if keep:
                raise _lib.OctmError(f"a contour has more than max_pts={out.max_pts} vertices; raise max_pts")
            if big >= MAX_MAX_PTS:
                raise _lib.OctmError(f"a contour has more than {MAX_MAX_PTS} vertices: pass a larger max_pts")
            big = min(big * 8, MAX_MAX_PTS)
        chunk = max(1, CONTOUR_CHUNK_BYTES // (k * 2 * big * 4 * 2))
        still = []
        for s0 in range(0, idx.numel(), chunk):
            sub = idx[s0:s0 + chunk]
            redo = _contour_chunk(yt[sub].contiguous(), yp[sub].contiguous(), k, big, out.mode, False, False,
                                  first_pos=None if first_pos is None else first_pos[sub].contiguous())
            for f in ("n_pts", "flags", "max_sq", "p95_sq", "sum_dist"):
                getattr(out, f)[sub] = getattr(redo, f)
            if out.mode == "first":
                still.append(sub[((redo.flags & over_bits) != 0).any(dim=1)])
        idx = torch.cat(still) if still else idx[:0]      # "all": no count exceeds the bound of this round
    return True


def derive_on_device(lp, ct, n, timers=None):
    """Float64 per-class metrics + this batch's dataset totals, computed by ``octm_derive_metrics``."""
    k, dev = lp.num_classes, lp.counts.device
    cls = torch.empty((n, k, len(_lib.CLASS_METRICS)), dtype=torch.float64, device=dev)
    bnd = torch.empty((n, k - 1, 3), dtype=torch.float64, device=dev) if lp.bnd_sq is not None else None
    tot = torch.empty((_lib.load().octm_totals_len(k),), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev), _Timed(timers, "derive"):
        _lib.call("octm_derive_metrics", _ptr(lp.counts), _ptr(lp.thick_absdiff), _ptr(lp.bnd_sq), _ptr(lp.bnd_abs),
                  _ptr(ct.n_pts) if ct else None, _ptr(ct.max_sq) if ct else None, _ptr(ct.p95_sq) if ct else None,
                  _ptr(ct.sum_dist) if ct else None, _ptr(ct.flags) if ct else None, n, lp.height, lp.width, k,
                  _ptr(cls), _ptr(bnd), _ptr(tot), _stream())
    return cls, bnd, tot


@dataclass
class SurfaceDiceOut:
    """Exact counts of the surface Dice pass (device tensors, uint32 stored as int32 bits)."""
    n_surf: torch.Tensor       # [N, K, 2]      (|V_t|, |V_p|): all-contour vertices of y_true / y_pred
    n_within: torch.Tensor     # [N, K, 2, T]   vertices within tolerance j of the other boundary; direction 0: pred -> true
    tolerances: tuple          # T tolerances in pixels, in the caller's order


def surface_dice(y_true, y_pred, num_classes, tolerances=(1.0,), *, timers=None):
    """Normalized surface Dice counts of every class at 1 to 4 tolerances ``0 <= tau <= 8`` pixels (build-defined,
    no reference counterpart; MONAI ``compute_surface_dice``, surface-distance ``compute_surface_dice_at_tolerance``).

    The surfaces are the whole boundaries, the all-contour vertex sets of ``contour_pass(mode="all")``; a vertex counts
    as within ``tau`` when the nearest vertex of the other map lies at ``sqrt(D2 / 4.0) <= tau``, the expression every
    contour distance of the suite is reported through.  One read of each label map (``octm_surface_dice_u8``).
    Tolerances may come in any order; the counts come back in that order.  ``derive.surface_dice`` turns them into
    float64 NSD values."""
    taus = derive.surface_dice_tolerances(tolerances)
    thr = [derive.surface_dice_threshold(t) for t in taus]
    order = sorted(range(len(taus)), key=lambda j: thr[j])
    yt, yp = _check_pair(y_true, y_pred)
    n, h, w = yt.shape
    k = int(num_classes)
    dev = yt.device
    n_surf = torch.empty((n, k, 2), dtype=torch.int32, device=dev)
    n_within = torch.empty((n, k, 2, len(taus)), dtype=torch.int32, device=dev)
    sorted_thr = (ctypes.c_uint32 * len(taus))(*[thr[j] for j in order])
    with torch.cuda.device(dev), _Timed(timers, "surface_dice"):
        _lib.call("octm_surface_dice_u8", _ptr(yt), _ptr(yp), n, h, w, k, sorted_thr, len(taus), _ptr(n_surf),
                  _ptr(n_within), _stream())
    if order != sorted(order):
        n_within = n_within[..., [order.index(j) for j in range(len(taus))]]
    return SurfaceDiceOut(n_surf, n_within, taus)


_surface_dice_pass = surface_dice      # evaluate()'s keyword argument of the same name shadows it there


@dataclass
class ComponentsOut:
    """Exact counts of the connected-component pass (device tensors, uint32 stored as int32 bits)."""
    n_comp: torch.Tensor       # [N, K, 2]   components of (y_true == c), (y_pred == c)
    n_hit: torch.Tensor        # [N, K, 2]   of those, the ones sharing a pixel with the other map's class c
    connectivity: int          # 4 or 8


def _connectivity(connectivity):
    if connectivity is True or connectivity is False or connectivity not in (4, 8):
        raise ValueError(f"components must be None, 4 or 8, got {connectivity!r}")
    return int(connectivity)


def components(y_true, y_pred, num_classes, connectivity=4, *, timers=None):
    """Connected components of every class of both maps (build-defined, no reference counterpart;
    ``scipy.ndimage.label`` at connectivity 4, ``skimage.measure.label``'s default at 8).

    ``n_comp[i, c, m]`` counts the components of ``(L_m == c)`` (m = 0: y_true, 1: y_pred) and ``n_hit[i, c, m]`` those
    of them that share at least one pixel with ``(L_o == c)`` of the other map: detected true lesions (m = 0) and
    matched predicted ones (m = 1).  Labels >= num_classes are never counted.  One row-streaming union-find per
    (item, map) (``octm_components_u8``), launched asynchronously on the current stream; ``derive.component_metrics``
    turns the counts into float64 scores."""
    conn = _connectivity(connectivity)
    yt, yp = _check_pair(y_true, y_pred)
    n, h, w = yt.shape
    k = int(num_classes)
    dev = yt.device
    n_comp = torch.empty((n, k, 2), dtype=torch.int32, device=dev)
    n_hit = torch.empty((n, k, 2), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev), _Timed(timers, "components"):
        _lib.call("octm_components_u8", _ptr(yt), _ptr(yp), n, h, w, k, conn, _ptr(n_comp), _ptr(n_hit), _stream())
    return ComponentsOut(n_comp, n_hit, conn)


_components_pass = components          # evaluate()'s keyword argument of the same name shadows it there


@dataclass
class SuiteResult:
    """Everything one evaluation produced, still on the device.

    ``class_metrics [N, K, 16]`` / ``boundary_metrics [N, K-1, 3]`` are the float64 scalars (column
    order ``_lib.CLASS_METRICS`` / ``_lib.BOUNDARY_METRICS``), ``totals`` the dataset-level partial sums
    of this batch.  ``metrics()`` copies them to the host; ``integers()`` the exact integer outputs."""
    num_items: int
    labels: LabelPassOut
    contours: ContourOut | None
    class_metrics: torch.Tensor | None = None
    boundary_metrics: torch.Tensor | None = None
    totals: torch.Tensor | None = None
    _inputs: tuple | None = field(default=None, repr=False)
    validate: bool = True
    _final: bool = field(default=False, repr=False)
    _host: dict | None = field(default=None, repr=False)
    _totals_host: np.ndarray | None = field(default=None, repr=False)
    contour_mode: str | None = "first"     # "first" / "all" (contour_pass modes), None without contour metrics
    surface: SurfaceDiceOut | None = None  # evaluate(surface_dice=...) only
    components: ComponentsOut | None = None  # evaluate(components=...) only

    @property
    def surface_dice_tolerances(self):
        """The tolerances (pixels) of ``metrics()["surface_dice"]``, or None when it was not requested."""
        return None if self.surface is None else self.surface.tolerances

    @property
    def component_connectivity(self):
        """The connectivity (4 or 8) of the component metrics, or None when they were not requested."""
        return None if self.components is None else self.components.connectivity

    def settle_overflow(self, vec):
        """Redo (with a larger vertex bound) this batch's items whose contour overflowed ``max_pts`` and
        recompute the epilogue; ``vec`` is the host copy of ``totals``.  No-op when nothing overflowed here.
        Returns True when something was redone."""
        if self.contours is None or self._final:
            return False
        self._final = True
        if not int(vec[-1]) & (_lib.CF_TRUE_OVERFLOW | _lib.CF_PRED_OVERFLOW):
            return False
        yt, yp = self._inputs
        _retry_overflow(self.contours, yt, yp, self.labels.num_classes, self.labels.first_pos)
        self.class_metrics, self.boundary_metrics, self.totals = derive_on_device(self.labels, self.contours, self.num_items)
        return True

    def totals_host(self):
        """The totals vector on the host (one small D2H).  Also where the two deferred checks happen: items with
        a label >= num_classes raise ValueError (``validate=True``), and items whose contour overflowed
        ``max_pts`` are redone before returning."""
        if self._totals_host is None:
            vec = self.totals.cpu().numpy()
            nb = int(_lib.load().octm_totals_sum_len(self.labels.num_classes))
            if self.validate and int(round(vec[nb - 1])) > 0:
                self._inputs = None
                raise ValueError(f"{int(round(vec[nb - 1]))} item(s) hold a label >= num_classes "
                                 f"{self.labels.num_classes}")
            if self.settle_overflow(vec):
                vec = self.totals.cpu().numpy()
            self._inputs = None
            self._totals_host = vec
        return self._totals_host

    def integers(self):
        """Host copies of the exact integer outputs (numpy; u64/u32 reinterpreted)."""
        self.totals_host()
        lp, ct = self.labels, self.contours
        d = {}
        if lp.counts is not None:
            d["confusion"] = lp.counts.cpu().numpy().view(np.uint64)
        if lp.thick_absdiff is not None:
            d["thickness_absdiff"] = lp.thick_absdiff.cpu().numpy()
            d["boundary_sq"] = lp.bnd_sq.cpu().numpy()
            d["boundary_abs"] = lp.bnd_abs.cpu().numpy()
        if lp.bnd_true is not None:
            d["boundary_true"] = lp.bnd_true.cpu().numpy()
            d["boundary_pred"] = lp.bnd_pred.cpu().numpy()
        if lp.first_pos is not None:
            d["first_pos"] = lp.first_pos.cpu().numpy().view(np.uint32)
        if lp.unsorted is not None:
            d["unsorted"] = lp.unsorted.cpu().numpy().view(np.uint32)
        if ct is not None:
            d["contour_n_pts"] = ct.n_pts.cpu().numpy().view(np.uint32)
            d["contour_flags"] = ct.flags.cpu().numpy().view(np.uint32)
            d["contour_max_sq"] = ct.max_sq.cpu().numpy().view(np.uint32)
            d["contour_p95_sq"] = ct.p95_sq.cpu().numpy().view(np.uint32)
            d["contour_sum_dist"] = ct.sum_dist.cpu().numpy()
        if self.surface is not None:
            d["surface_dice_n_surf"] = self.surface.n_surf.cpu().numpy().view(np.uint32)
            d["surface_dice_n_within"] = self.surface.n_within.cpu().numpy().view(np.uint32)
        if self.components is not None:
            d["component_count"] = self.components.n_comp.cpu().numpy().view(np.uint32)
            d["component_hits"] = self.components.n_hit.cpu().numpy().view(np.uint32)
        return d

    def metrics(self):
        """float64 ``[N, K]`` (``[N, K-1]`` for boundary errors) arrays keyed by reference function name,
        as computed on the device."""
        if self._host is None:
            self.totals_host()
            cls = self.class_metrics.cpu().numpy()
            m = {name: cls[:, :, i] for i, name in enumerate(_lib.CLASS_METRICS)}
            if self.contours is None:
                for name in ("hausdorff_distance", "hausdorff_distance_95", "assd"):
                    m.pop(name)
            else:
                m["contour_valid"] = ~np.isnan(m["hausdorff_distance"])
            if self.labels.thick_absdiff is None:
                m.pop("thickness_difference")
            if self.boundary_metrics is not None:
                b = self.boundary_metrics.cpu().numpy()
                m.update({name: b[:, :, i] for i, name in enumerate(_lib.BOUNDARY_METRICS)})
            if self.surface is not None:        # a ratio of exact counts, evaluated on the host
                m["surface_dice"] = derive.surface_dice(self.surface.n_surf.cpu().numpy().view(np.uint32),
                                                        self.surface.n_within.cpu().numpy().view(np.uint32))
            if self.components is not None:     # ratios of exact counts, evaluated on the host
                m.update(derive.component_metrics(self.components.n_comp.cpu().numpy().view(np.uint32),
                                                  self.components.n_hit.cpu().numpy().view(np.uint32)))
            self._host = m
        return self._host

    def metrics_host(self):
        """The same scalars re-derived on the host from the integer outputs (``derive.py``); the two
        agree bit for bit (tests/test_gpu_derive.py)."""
        ints = self.integers()
        m = {}
        if "confusion" in ints:
            m.update(derive.count_metrics(*derive.class_counts(ints["confusion"])))
        if "thickness_absdiff" in ints:
            m["thickness_difference"] = derive.thickness_difference(ints["thickness_absdiff"], self.labels.width)
            m.update(derive.boundary_errors(ints["boundary_sq"], ints["boundary_abs"], self.labels.width))
        if "contour_n_pts" in ints:
            m.update(derive.contour_metrics(ints["contour_n_pts"], ints["contour_max_sq"],
                                            ints["contour_p95_sq"], ints["contour_sum_dist"]))
        if "surface_dice_n_surf" in ints:
            m["surface_dice"] = derive.surface_dice(ints["surface_dice_n_surf"], ints["surface_dice_n_within"])
        if "component_count" in ints:
            m.update(derive.component_metrics(ints["component_count"], ints["component_hits"]))
        return m


def _contour_mode(contours):
    if not isinstance(contours, str):
        return "first" if contours else None
    if contours not in CONTOUR_MODES:
        raise ValueError(f"contours must be True, False, 'first' or 'all', got {contours!r}")
    return contours


def evaluate(y_true, y_pred, num_classes, *, contours=True, boundaries=False, max_pts=None, timers=None,
             validate=True, surface_dice=None, components=None):
    """The full suite on a batch of label maps: fused label pass, contour kernels, float64 epilogue.

    ``contours``: ``True`` / ``"first"`` = hausdorff / hd95 / assd on contour ``[0]`` of each class mask, as the
    reference computes them; ``"all"`` = on every contour of each class (the whole boundary, see ``contour_pass``);
    ``False`` = no contour metrics.

    ``surface_dice``: ``None`` (default, nothing extra runs) or a tolerance or 1 to 4 tolerances in pixels
    (``0 <= tau <= 8``): adds ``metrics()["surface_dice"]``, float64 ``[N, K, T]``, the normalized surface Dice of the
    whole boundary of each class at each tolerance (see ``surface_dice``; independent of ``contours``), the counts
    ``integers()["surface_dice_n_surf"]`` / ``["surface_dice_n_within"]`` and ``surface_dice_tolerances``.

    ``components``: ``None`` (default, nothing extra runs) or the connectivity 4 or 8: adds the float64 ``[N, K]``
    ``metrics()`` ``component_count_error``, ``component_recall``, ``component_precision`` and ``component_f1`` of the
    connected components of each class (see ``components`` and ``derive.component_metrics``; independent of
    ``contours`` and ``surface_dice``), the counts ``integers()["component_count"]`` / ``["component_hits"]``
    (uint32 ``[N, K, 2]``) and ``component_connectivity``.

    Everything is launched asynchronously on the current stream; nothing is read back until
    ``totals_host()`` / ``metrics()`` / ``integers()`` is called on the result.
    ``timers``: optional dict filled with (start, end) CUDA-event pairs per kernel family.
    ``validate``: a label >= num_classes (an ignore label such as 255, a wrong class count) raises ValueError when
    the results are read.  The check costs nothing extra: the label pass never aliases such a pixel into another
    class but drops it, so the item's confusion counts do not add up to H * W, which the totals kernel counts."""
    mode = _contour_mode(contours)
    taus = None if surface_dice is None else derive.surface_dice_tolerances(surface_dice)
    conn = None if components is None else _connectivity(components)
    yt, yp = _check_pair(y_true, y_pred)
    first = mode == "first"
    # contour [0] is seeded by the label pass, and its boundary rows and certificate skip the walk on layered maps
    lp = label_pass(yt, yp, num_classes, counts=True, columns=True, seeds=first, boundaries=boundaries or first,
                    timers=timers, certify=first)
    sd = None if taus is None else _surface_dice_pass(yt, yp, num_classes, taus, timers=timers)
    cc = None if conn is None else _components_pass(yt, yp, num_classes, conn, timers=timers)
    ct = None
    if mode is not None:
        ct = contour_pass(yt, yp, num_classes, lp.first_pos, max_pts=max_pts, timers=timers, check_overflow=False,
                          boundaries=(lp.bnd_true, lp.bnd_pred) if first else None,
                          unsorted=lp.unsorted if first else None, mode=mode)
        if first and not boundaries:
            lp.bnd_true = lp.bnd_pred = None
    cls, bnd, tot = derive_on_device(lp, ct, yt.shape[0], timers)
    return SuiteResult(yt.shape[0], lp, ct, cls, bnd, tot, (yt, yp) if ct is not None else None,
                       validate=bool(validate), contour_mode=mode, surface=sd, components=cc)


def _cat_results(parts):
    def cat(objs, f):
        vals = [getattr(o, f) for o in objs]
        return None if vals[0] is None else torch.cat(vals)
    for p in parts:
        p.totals_host()                       # settles any overflow retry per chunk
    lps = [p.labels for p in parts]
    lp = LabelPassOut(lps[0].num_classes, lps[0].height, lps[0].width,
                      *[cat(lps, f) for f in ("counts", "thick_absdiff", "bnd_sq", "bnd_abs", "bnd_true", "bnd_pred",
                                              "first_pos", "unsorted")])
    ct = None
    if parts[0].contours is not None:
        cts = [p.contours for p in parts]
        ct = ContourOut(*[cat(cts, f) for f in ("n_pts", "flags", "max_sq", "p95_sq", "sum_dist")], None, None,
                        cts[0].max_pts, cts[0].mode)
    n = sum(p.num_items for p in parts)
    cls, bnd, tot = derive_on_device(lp, ct, n)            # per-item values again + totals of the whole batch
    sd = None
    if parts[0].surface is not None:
        sds = [p.surface for p in parts]
        sd = SurfaceDiceOut(cat(sds, "n_surf"), cat(sds, "n_within"), sds[0].tolerances)
    cc = None
    if parts[0].components is not None:
        ccs = [p.components for p in parts]
        cc = ComponentsOut(cat(ccs, "n_comp"), cat(ccs, "n_hit"), ccs[0].connectivity)
    res = SuiteResult(n, lp, ct, cls, bnd, tot, validate=parts[0].validate, contour_mode=parts[0].contour_mode,
                      surface=sd, components=cc)
    res._final = True
    return res


_PINNED = {}       # nbytes class -> grow-only pinned host staging buffer of evaluate_host(pack=True)


def _pinned(nbytes):
    buf = _PINNED.get("buf")
    if buf is None or buf.numel() < nbytes:
        _PINNED.pop("buf", None)
        buf = torch.empty((nbytes,), dtype=torch.uint8, pin_memory=True)
        _PINNED["buf"] = buf
    return buf


def evaluate_host(y_true, y_pred, num_classes, *, contours=True, device=None, chunk_items=None,
                  max_pts=None, pack=False, pack_threads=0, validate=True, surface_dice=None, components=None):
    """The full suite on HOST label maps (numpy arrays or CPU torch tensors, ideally pinned).

    Items are streamed to the GPU in chunks through two staging buffers: the host->device copy of
    chunk i+1 (copy stream) overlaps the kernels of chunk i (compute stream).  The path is bound by the
    PCIe copy (~50 GB/s).  ``pack=True`` (``num_classes <= 16``) sends the labels two per byte: the host
    packs a chunk into pinned memory (``octm_host_pack_nibbles``, all cores) while the previous chunk is
    being copied, and a streaming kernel expands it in HBM.  Off by default: on the 16-core B200 boxes the
    packer sustains ~80 GB/s of input, which only ties with the plain copy (measured 92-100 k vs 98-100 k
    B-scans/s); it pays on hosts with more memory bandwidth per PCIe lane.  Results stay on the device
    until ``metrics()`` / ``integers()`` reads them back."""
    if not torch.cuda.is_available():
        raise RuntimeError("a CUDA device is required: this package has no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    to_t = lambda a: a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))   # noqa: E731
    ht, hp = to_t(y_true), to_t(y_pred)
    if ht.is_cuda or hp.is_cuda:
        raise TypeError("evaluate_host takes host arrays; use evaluate() for CUDA tensors")
    if ht.dtype == torch.bool:
        ht, hp = ht.view(torch.uint8), hp.view(torch.uint8)
    if ht.dtype != torch.uint8 or hp.dtype != torch.uint8:
        raise TypeError("label maps must be uint8")
    if ht.shape != hp.shape or ht.dim() != 3:
        raise ValueError("expected two [N, H, W] arrays of equal shape")
    ht, hp = ht.contiguous(), hp.contiguous()
    n, h, w = ht.shape
    use_pack = (bool(pack) if pack != "auto" else True) and int(num_classes) <= 16
    if chunk_items is None:
        chunk_items = max(1, min(n, (256 << 20) // max(1, h * w)))       # ~256 MiB per map per buffer
    per_map = chunk_items * h * w
    half = (per_map + 1) // 2
    half_al = (half + 255) & ~255
    with torch.cuda.device(dev):
        compute = torch.cuda.current_stream()
        copy, flat = _staging(dev, 4 * per_map + (4 * half_al if use_pack else 0))
        copy.wait_stream(compute)           # earlier users of the (cached) staging buffers are done
        views = flat[:4 * per_map].view(4, chunk_items, h, w)
        bufs = [(views[0], views[1]), (views[2], views[3])]
        if use_pack:
            dpk = flat[4 * per_map:4 * per_map + 4 * half_al].view(4, half_al)
            hpk = _pinned(4 * half_al)[:4 * half_al].view(4, half_al)
            h2d_done = [None, None]
            lib = _lib.load()
        freed = [None, None]
        starts = list(range(0, n, chunk_items))
        ready = {}

        def issue_copy(ci):
            s0, e0 = starts[ci], min(n, starts[ci] + chunk_items)
            bt, bp = bufs[ci & 1]
            if use_pack:
                b = ci & 1
                if h2d_done[b] is not None:
                    h2d_done[b].synchronize()                    # the pinned half-buffers of chunk ci-2 have been sent
                m = (e0 - s0) * h * w
                for k, src in ((0, ht), (1, hp)):
                    rc = lib.octm_host_pack_nibbles(src[s0:e0].data_ptr(), hpk[2 * b + k].data_ptr(), m, int(pack_threads))
                    if rc != 0:
                        raise _lib.OctmError("octm_host_pack_nibbles failed")
            with torch.cuda.stream(copy):
                if freed[ci & 1] is not None:
                    copy.wait_event(freed[ci & 1])               # kernels of chunk ci-2 are done with it
                if use_pack:
                    nb = (m + 1) // 2
                    dpk[2 * b][:nb].copy_(hpk[2 * b][:nb], non_blocking=True)
                    dpk[2 * b + 1][:nb].copy_(hpk[2 * b + 1][:nb], non_blocking=True)
                    h2d_done[b] = torch.cuda.Event()
                    h2d_done[b].record(copy)
                else:
                    bt[:e0 - s0].copy_(ht[s0:e0], non_blocking=True)
                    bp[:e0 - s0].copy_(hp[s0:e0], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            ready[ci] = ev

        def expand(ci):
            """compute stream: packed chunk -> uint8 labels in the chunk's device buffers"""
            s0, e0 = starts[ci], min(n, starts[ci] + chunk_items)
            m = (e0 - s0) * h * w
            b = ci & 1
            for k in (0, 1):
                _lib.call("octm_unpack_nibbles_u8", _ptr(dpk[2 * b + k]), m, _ptr(bufs[b][k]), _stream())

        parts = []
        issue_copy(0)
        for ci, s0 in enumerate(starts):
            e0 = min(n, s0 + chunk_items)
            if ci >= 1:
                # chunk ci-1 still owns the staging buffer the next copy overwrites: settle it first (its
                # overflow retry, if any, re-reads its inputs).  One ~1 KB read-back per chunk.
                parts[ci - 1].totals_host()
            if ci + 1 < len(starts):
                issue_copy(ci + 1)                               # overlaps the kernels launched below
            bt, bp = bufs[ci & 1]
            compute.wait_event(ready.pop(ci))
            if use_pack:
                expand(ci)
            parts.append(evaluate(bt[:e0 - s0], bp[:e0 - s0], num_classes, contours=contours, max_pts=max_pts,
                                  validate=validate, surface_dice=surface_dice, components=components))
            done = torch.cuda.Event()
            done.record(compute)
            freed[ci & 1] = done
        parts[-1].totals_host()        # the staging buffers are shared with later calls: settle before returning
        return parts[0] if len(parts) == 1 else _cat_results(parts)


def labels_from_scores(scores, *, channels_last=False, out=None):
    """Model scores -> ``uint8`` label map: argmax over the class dimension (SURVEY.md 8f rank 1).

    ``scores``: CUDA float32 / float16 / bfloat16 tensor ``[N, K, H, W]`` (what every model of the
    reference returns) or ``[N, H, W, K]`` with ``channels_last=True``; logits or probabilities alike.
    Ties go to the first maximal class and a NaN counts as maximal, as in numpy / torch ``argmax``."""
    if not isinstance(scores, torch.Tensor) or not scores.is_cuda:
        raise TypeError("scores must be a CUDA torch tensor")
    if scores.dim() != 4:
        raise ValueError("expected [N, K, H, W] (or [N, H, W, K] with channels_last=True) scores")
    dt = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}.get(scores.dtype)
    if dt is None:
        raise TypeError(f"scores must be float32, float16 or bfloat16, got {scores.dtype}")
    s = scores.contiguous()
    if channels_last:
        n, h, w, k = s.shape
    else:
        n, k, h, w = s.shape
    if k > 256:
        raise ValueError("more than 256 classes do not fit a uint8 label map")
    if out is None:
        out = torch.empty((n, h, w), dtype=torch.uint8, device=s.device)
    elif out.shape != (n, h, w) or out.dtype != torch.uint8 or not out.is_contiguous() or out.device != s.device:
        raise ValueError("out must be a contiguous uint8 [N, H, W] tensor on the scores' device")
    with torch.cuda.device(s.device):
        _lib.call("octm_argmax_labels", _ptr(s), dt, n, k, h * w, 1 if channels_last else 0, _ptr(out), _stream())
    return out


def evaluate_scores(y_true, scores, num_classes=None, *, channels_last=False, **kw):
    """``evaluate(y_true, argmax(scores), ...)`` with the argmax done by ``labels_from_scores``."""
    k = scores.shape[-1 if channels_last else 1] if num_classes is None else int(num_classes)
    return evaluate(y_true, labels_from_scores(scores, channels_last=channels_last), k, **kw)


def auc_scores(y_true, scores, *, single_class_value=float("nan")):
    """Per-item area under the ROC curve (``auc_score`` of the reference, batched): float64 ``[N]``.

    ``y_true``: CUDA uint8 / bool ``[N, ...]`` binary masks; ``scores``: CUDA float16 / bfloat16 /
    float32 / float64 tensor of the same shape.  Each item is flattened, as the reference does."""
    for name, t in (("y_true", y_true), ("scores", scores)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise TypeError(f"{name} must be a CUDA torch tensor")
    if y_true.dtype not in (torch.uint8, torch.bool):
        raise TypeError("y_true must be uint8 or bool")
    dt = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16,
          torch.float64: _lib.DTYPE_F64}.get(scores.dtype)
    if dt is None:
        raise TypeError(f"scores must be a floating tensor, got {scores.dtype}")
    if y_true.shape != scores.shape:
        raise ValueError(f"shape mismatch: {tuple(y_true.shape)} vs {tuple(scores.shape)}")
    yt = (y_true.view(torch.uint8) if y_true.dtype == torch.bool else y_true).contiguous()
    sc = scores.contiguous()
    n = yt.shape[0]
    elems = yt[0].numel() if n else 0
    out = torch.empty((n,), dtype=torch.float64, device=yt.device)
    if n == 0:
        return out
    with torch.cuda.device(yt.device):
        nbytes = int(_lib.load().octm_auc_workspace_bytes(n, elems, dt))
        ws = _vertex_scratch(yt.device, (nbytes + 3) // 4 + 64)
        _lib.call("octm_auc_u8", _ptr(yt), _ptr(sc), dt, n, elems, float(single_class_value), _ptr(out), _ptr(ws),
                  ws.numel() * 4, _stream())
    return out


def surface_distance_3d(vol_true, vol_pred, num_classes, *, units=None):
    """3-D surface-distance integers per class of two label volumes ``[D0, D1, D2]`` (BASELINE config 5).

    Surfaces = region voxels with a 6-neighbour outside the region; exact squared Euclidean distances by
    a separable distance transform.  ``units=(begin, end)`` restricts the work to a range of the
    ``2 * num_classes`` (class, direction) units (multi-GPU sharding; the other entries stay zero and
    the per-rank outputs add up).  Returns a dict of CUDA tensors ``n_pts [K, 2]``, ``max_sq [K, 2]``,
    ``p95_sq [K, 2, 2]``, ``sum_dist [K, 2]``; ``surface_metrics_3d`` turns them into hd / hd95 / assd."""
    for name, t in (("vol_true", vol_true), ("vol_pred", vol_pred)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype not in (torch.uint8, torch.bool) or t.dim() != 3:
            raise TypeError(f"{name} must be a CUDA uint8 tensor [D0, D1, D2]")
    if vol_true.shape != vol_pred.shape:
        raise ValueError("shape mismatch")
    vt = (vol_true.view(torch.uint8) if vol_true.dtype == torch.bool else vol_true).contiguous()
    vp = (vol_pred.view(torch.uint8) if vol_pred.dtype == torch.bool else vol_pred).contiguous()
    d0, d1, d2 = vt.shape
    k = int(num_classes)
    ub, ue = (0, 2 * k) if units is None else (int(units[0]), int(units[1]))
    dev = vt.device
    out = {"n_pts": torch.zeros((k, 2), dtype=torch.int32, device=dev),
           "max_sq": torch.zeros((k, 2), dtype=torch.int32, device=dev),
           "p95_sq": torch.zeros((k, 2, 2), dtype=torch.int32, device=dev),
           "sum_dist": torch.zeros((k, 2), dtype=torch.float64, device=dev)}
    with torch.cuda.device(dev):
        nbytes = int(_lib.load().octm_surface3d_workspace_bytes(d0, d1, d2))
        ws = _vertex_scratch(dev, (nbytes + 3) // 4 + 64)
        _lib.call("octm_surface3d_u8", _ptr(vt), _ptr(vp), d0, d1, d2, k, ub, ue, _ptr(out["n_pts"]), _ptr(out["max_sq"]),
                  _ptr(out["p95_sq"]), _ptr(out["sum_dist"]), _ptr(ws), ws.numel() * 4, _stream())
    return out


def surface_metrics_3d(ints):
    """hausdorff_distance / hausdorff_distance_95 / assd per class from ``surface_distance_3d`` outputs
    (after any cross-rank sum), with the reference's 2-D definitions carried over to voxel surfaces."""
    g = lambda key: ints[key].cpu().numpy() if isinstance(ints[key], torch.Tensor) else np.asarray(ints[key])   # noqa: E731
    return derive.contour_metrics(g("n_pts").view(np.uint32), g("max_sq").view(np.uint32), g("p95_sq").view(np.uint32),
                                  g("sum_dist"), lattice=1.0)


def validate_labels(labels, num_classes):
    """Raise ValueError if any label is >= num_classes (one reduction kernel + a 4-byte readback)."""
    t = (labels.view(torch.uint8) if labels.dtype == torch.bool else labels).contiguous()
    out = torch.zeros(1, dtype=torch.int32, device=t.device)
    with torch.cuda.device(t.device):
        _lib.call("octm_validate_labels_u8", _ptr(t), t.numel(), _ptr(out), _stream())
    mx = int(out.item())
    if mx >= num_classes:
        raise ValueError(f"label {mx} >= num_classes {num_classes}")
