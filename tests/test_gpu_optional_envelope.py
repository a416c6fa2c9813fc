"""GPU parity of the optional passes with the fast exact oracles (``envelope_oracle``) at the geometry envelope:
``contour_pass(mode="all")`` (``contour_all_vertices_kernel``), ``surface_dice`` (``surface_dice_kernel``),
``components`` (``components_kernel``) and ``spacing=`` (``distance_spacing_kernel``, ``octm_surface_dice_spacing_u8``)
on tall maps of 4095 to 8192 rows, wide maps of 2056 to 8192 columns, 15 and 16 classes, contours of 8192 to 40000
vertices, batches with more units than resident CTAs, and sides of 8193 that must be refused.

The kernels route on shapes and device data, so no route is observable from outside; every case asserts instead the
input property that forces its route (row count, width and alignment, class groups, vertex counts, units per grid),
so that a change of the inputs cannot silently move a case off its branch.  Integer counts, ``d2`` and the order
statistics are compared bit for bit, ``sum_dist`` within 1e-12."""
import math

import numpy as np
import pytest
import torch

from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, derive, suite, synth

import envelope_oracle as eo
import geometry_oracle as go

pytestmark = pytest.mark.gpu

OCT = (0.0039, 0.0117)                       # mm: axial (rows), lateral (columns)
PIX_TAUS = (0.0, 1.0, math.sqrt(5.0) / 2, 8.0)
SP_TILE = 16384                              # distance_spacing_kernel: source vertices per sorted tile
SP_QUERIES = 8192                            # distance_spacing_kernel: queries whose d2 stay in shared memory
SD_WARPS, SD_SEG, SD_MAX_REACH = 8, 512, 16  # surface_dice_kernel: rows per iteration, columns per pass, reach
MAX_BLOCKS_PER_SM = 32                       # sm_100


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _sp_taus(spacing):
    lim = derive.surface_dice_spacing_limit(spacing)
    return (0.0, lim / 4, lim / 2, lim)


def _profiled(fn):
    with _lib.kernel_profile() as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, prof.kernels


# ------------------------------------------------------------------------------------------------------ checkers
def check_contours(yt, yp, k, out, mode, spacing=None, items=None):
    """``contour_pass`` output against the oracle; result item ``items[j]`` (default j) is ``yt[j]`` / ``yp[j]``.
    Returns the per-unit (item, class, direction) (ns, nq) vertex counts the search saw."""
    n_pts = _u32(out.n_pts)
    conv = _u32 if spacing is None else (lambda t: t.cpu().numpy())
    max_sq, p95, sums = conv(out.max_sq), conv(out.p95_sq), out.sum_dist.cpu().numpy()
    verts = None if out.verts is None else _u32(out.verts)
    sq = None if out.sq is None else conv(out.sq)
    counts = []
    items = range(len(yt)) if items is None else items
    for j, i in enumerate(items):
        for c, (vt, vp, d) in enumerate(eo.contours(yt[j], yp[j], k, mode, spacing)):
            where = (i, c)
            assert tuple(int(v) for v in n_pts[i, c]) == (len(vt), len(vp)), (where, n_pts[i, c])
            if d is None:
                continue
            got = None
            if verts is not None:
                got = [verts[i, c, s, :n_pts[i, c, s]] for s in (0, 1)]
                got = [np.stack([g >> 16, g & 0xffff], axis=1).astype(np.int64) for g in got]
                for g, ref in zip(got, (vt, vp)):
                    if mode == "all":
                        np.testing.assert_array_equal(g, ref, err_msg=str(where))       # raster order
                    else:
                        assert sorted(map(tuple, g)) == sorted(map(tuple, ref)), where  # contour order of the walk
            for di in (0, 1):
                want = d[di]
                if sq is not None:
                    if mode == "first":      # the stored d2 follow the walk's vertex order
                        want = eo.distances(got[di], got[1 - di], spacing)
                    assert np.array_equal(sq[i, c, di, :len(want)], want), (where, di)
                vmax, lo_, hi_, s = eo.order_stats(want)
                assert max_sq[i, c, di] == vmax, (where, di, max_sq[i, c, di], vmax)
                assert (p95[i, c, di, 0], p95[i, c, di, 1]) == (lo_, hi_), (where, di)
                np.testing.assert_allclose(sums[i, c, di], s, rtol=1e-12, atol=0, err_msg=str((where, di)))
                counts.append((len(d[1 - di]), len(want)))      # (ns: the other direction's queries, nq)
    return counts


def check_surface(yt, yp, k, taus, sd, spacing=None, items=None):
    n_surf, n_within = _u32(sd.n_surf), _u32(sd.n_within)
    items = range(len(yt)) if items is None else items
    for j, i in enumerate(items):
        ns, nw = eo.surface_counts(yt[j], yp[j], k, taus, spacing)
        assert np.array_equal(n_surf[i], ns), i
        assert np.array_equal(n_within[i], nw), i


def check_components(yt, yp, k, conn, cc, items=None):
    n_comp, n_hit = _u32(cc.n_comp), _u32(cc.n_hit)
    items = range(len(yt)) if items is None else items
    for j, i in enumerate(items):
        nc, nh = eo.component_counts(yt[j], yp[j], k, conn)
        assert np.array_equal(n_comp[i], nc), (i, n_comp[i], nc)
        assert np.array_equal(n_hit[i], nh), (i, n_hit[i], nh)


def run_every_pass(yt, yp, k, t, p, spacing_modes=("all", "first")):
    """Each optional pass on the device pair (t, p) against the oracle of the host pair (yt, yp)."""
    check_contours(yt, yp, k, suite.contour_pass(t, p, k, mode="all"), "all")
    check_surface(yt, yp, k, PIX_TAUS, suite.surface_dice(t, p, k, PIX_TAUS))
    for conn in (4, 8):
        check_components(yt, yp, k, conn, suite.components(t, p, k, conn))
    for mode in spacing_modes:
        out, kernels = _profiled(lambda: suite.contour_pass(t, p, k, mode=mode, spacing=OCT))
        assert "distance_spacing_kernel" in kernels
        check_contours(yt, yp, k, out, mode, OCT)
    check_surface(yt, yp, k, _sp_taus(OCT), suite.surface_dice(t, p, k, _sp_taus(OCT), spacing=OCT), OCT)


def _groups(w, k, reach, cuda):
    """surface_dice_kernel's class groups, restated from the host code: (n_groups, group, classes of the last group)."""
    halo = (reach + 1) // 2
    slots = SD_WARPS + 2 * halo
    nw = (w + SD_SEG - 1) // SD_SEG * 32
    per_class = slots * 2 * (nw + 2) * 4
    budget = torch.cuda.get_device_properties(cuda).shared_memory_per_block_optin - 4096
    group = min(budget // per_class, k)
    n_groups = -(-k // group)
    group = -(-k // n_groups)
    return n_groups, group, k - (n_groups - 1) * group


# ------------------------------------------------------------------------------------------------- A. tall maps
def _tall_items(h, w, k, seed, cuda):
    yt, yp = synth.layered_pair(2, h, w, k, seed=seed)
    yp[1] = synth.layered_pair(2, h, w, k, seed=seed, noise=2e-3)[1][1]
    rt, rp = synth.ragged_pair_device(1, h, w, k, seed=seed + 1, device=cuda)
    return np.concatenate([yt, rt.cpu().numpy()]), np.concatenate([yp, rp.cpu().numpy()])


@pytest.mark.parametrize("h,w,k", [(4095, 64, 4), (4096, 16, 6), (4097, 64, 5), (8192, 16, 3), (8192, 64, 6)])
def test_tall_maps(cuda, h, w, k):
    """Clean, noisy (2e-3) and ragged items: the surface Dice ring wraps hundreds of times, packed vertex rows reach
    y2 = 2 H - 2, and the components of every layer stay open through all rows."""
    yt, yp = _tall_items(h, w, k, 4000 + h + w + k, cuda)
    yp[0, h - 1, w // 2] = 0                         # a crack in the last row: packed vertex row y2 = 2 H - 2
    assert h > 4094 and (np.diff(yp[1].astype(np.int16), axis=0) < 0).any()       # the noisy item is out of order
    v = eo.contours(yt[0], yp[0], k, "all")
    assert max(int(vp[:, 0].max()) for _, vp, _ in v if len(vp)) == 2 * h - 2
    nc, _ = eo.component_counts(yt[0], yp[0], k, 4)
    assert (nc[:, 0] == 1).all()                     # clean layers: each class one component from its top to its bottom
    run_every_pass(yt, yp, k, _dev(yt, cuda), _dev(yp, cuda))


def test_serpentine_component_through_8192_rows(cuda):
    """One component of class 1 that winds through every row of an 8192 x 16 map (4- and 8-connected); the prediction
    is cut once, into two."""
    h, w = 8192, 16
    yt = np.zeros((h, w), np.uint8)
    yt[0::2, 1:w - 1] = 1
    yt[1::4, w - 2] = 1
    yt[3::4, 1] = 1
    yp = yt.copy()
    yp[4000, 1:w - 1] = 0
    yp[4000, 0] = 2
    yt, yp = yt[None], yp[None]
    for conn in (4, 8):
        nc, nh = eo.component_counts(yt[0], yp[0], 3, conn)
        assert nc[1].tolist() == [1, 2] and nh[1].tolist() == [1, 2], conn
        check_components(yt, yp, 3, conn, suite.components(_dev(yt, cuda), _dev(yp, cuda), 3, conn))
    assert (yt[0] == 1).any(axis=1).all()


# ------------------------------------------------------------------------------------------------- B. wide maps
@pytest.mark.parametrize("h,w,k,misaligned", [(64, 2056, 5, False), (48, 4096, 16, False), (16, 8191, 3, False),
                                              (48, 8192, 16, False), (32, 8192, 5, True)])
def test_wide_maps(cuda, h, w, k, misaligned):
    """W % 16 == 0 on 16-byte aligned maps takes the 16-byte loaders, anything else the byte-wise ones."""
    yt, yp = synth.layered_pair(2, h, w, k, seed=h + w + k, noise=2e-3, min_gap=1 if k > 8 else 2)
    yt[1], _ = synth.layered_pair(1, h, w, k, seed=h + w + k + 1, min_gap=1 if k > 8 else 2)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    if misaligned:
        bufs = [torch.empty(a.size + 1, dtype=torch.uint8, device=cuda) for a in (yt, yp)]
        t, p = [b[1:].view(a.shape).copy_(torch.from_numpy(a)) for a, b in zip((yt, yp), bufs)]
    vec = w % 16 == 0 and t.data_ptr() % 16 == 0 and p.data_ptr() % 16 == 0
    assert vec == (w in (4096, 8192) and not misaligned)
    run_every_pass(yt, yp, k, t, p)


@pytest.mark.parametrize("kind", ["checkerboard", "random_rows"])
def test_components_one_run_per_pixel(cuda, kind):
    """At W = 8192 every row is W runs (ncur == W, the sentinel at index W): the largest run state the kernel has."""
    h, w, k = 16, 8192, 3
    rng = np.random.default_rng(8192)
    if kind == "checkerboard":
        yt = ((np.arange(h)[:, None] + np.arange(w)[None, :]) % 2).astype(np.uint8)[None]
    else:       # uniform random labels with no two equal neighbours in a row
        step = rng.integers(1, k, size=(1, h, w))
        yt = (np.cumsum(step, axis=2) % k).astype(np.uint8)
    yp = (np.cumsum(rng.integers(1, k, size=(1, h, w)), axis=2) % k).astype(np.uint8)
    for a in (yt, yp):
        assert (a[0, :, 1:] != a[0, :, :-1]).all()                  # a run starts at every pixel
    for conn in (4, 8):
        check_components(yt, yp, k, conn, suite.components(_dev(yt, cuda), _dev(yp, cuda), k, conn))
    if kind == "checkerboard":
        assert eo.component_counts(yt[0], yp[0], k, 4)[0][0, 0] == h * w // 2
        assert eo.component_counts(yt[0], yp[0], k, 8)[0][0, 0] == 1


@pytest.mark.parametrize("k", [16, 5])
@pytest.mark.parametrize("spacing", [None, OCT])
def test_surface_dice_class_groups(cuda, k, spacing):
    """tau at the kernel's reach of 16 lattice rows: one class's ring at W = 8192 is ~98.7 KB, so the classes split
    into groups of 2; at K = 5 the last group holds one class."""
    h, w = 40, 8192
    if spacing is None:
        taus = (1.0, 8.0)
        reach = max(a for a in range(SD_MAX_REACH + 1) if a * a <= derive.surface_dice_threshold(8.0))
    else:
        taus = (OCT[0], derive.surface_dice_spacing_limit(OCT))
        wy = OCT[0] ** 2
        reach = max(a for a in range(SD_MAX_REACH + 1) if math.sqrt(wy * (a * a) / 4.0) <= taus[-1])
    assert reach == SD_MAX_REACH
    n_groups, group, last = _groups(w, k, reach, cuda)
    assert n_groups > 1 and group == 2 and (last < group) == (k == 5)
    yt, yp = synth.layered_pair(3, h, w, k, seed=77 + k, noise=2e-3, min_gap=1 if k > 8 else 2)
    sd = suite.surface_dice(_dev(yt, cuda), _dev(yp, cuda), k, taus, spacing=spacing)
    check_surface(yt, yp, k, taus, sd, spacing)


# ----------------------------------------------------------------------------------------- C. spacing search routes
def _long_short_pair(n_long, h, w):
    """A true boundary of exactly ``n_long`` vertices (sawtooth) against a predicted flat one of W vertices."""
    yt, _ = go.sawtooth_pair(h, w, n_long, 0)
    yp = np.broadcast_to(np.arange(h)[:, None] >= h // 2, (h, w)).astype(np.uint8)[None]
    return yt, yp


@pytest.mark.parametrize("mode", ["all", "first"])
@pytest.mark.parametrize("case", ["8192", "8193", "16384", "16385", "40000", "long_short"])
def test_spacing_search_routes(cuda, case, mode):
    """Queries in shared memory (nq <= 8192, d2 not kept) or in global d2 (nq > 8192, or d2 kept); sources in one sorted
    tile (ns <= 16384) or several (ns > 16384 needs max_pts > 16384), each later tile resuming from the d2 so far."""
    h, w = 128, 1024
    if case == "long_short":
        yt, yp = _long_short_pair(20000, h, w)
    else:
        yt, yp = go.sawtooth_pair(h, w, int(case), 1)
    counts = [(len(vt), len(vp)) for vt, vp, _ in eo.contours(yt[0], yp[0], 2, mode)]
    longest = max(max(c) for c in counts)
    max_pts = (max(longest, 8) + 3) & ~3
    if case != "long_short":
        assert counts[0] == (int(case), int(case)) or mode == "first" and counts[0][0] == int(case)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    for keep in (False, True):
        out, kernels = _profiled(lambda: suite.contour_pass(t, p, 2, mode=mode, spacing=OCT, max_pts=max_pts,
                                                            return_vertices=keep, return_sq=keep))
        assert "distance_spacing_kernel" in kernels
        units = check_contours(yt, yp, 2, out, mode, OCT)
        tile = min(max_pts, SP_TILE)
        qcap = 0 if keep else min(max_pts, SP_QUERIES)
        routes = {(ns > tile, nq > qcap) for ns, nq in units}
        if case == "8192":
            assert (keep or routes == {(False, False)}) and longest == 8192
        elif case in ("8193", "16384"):
            assert (False, True) in routes
        elif case in ("16385", "40000"):
            assert (True, True) in routes and max_pts > SP_TILE
            if case == "40000":
                assert longest > 2 * SP_TILE
        else:
            assert (True, keep) in routes and (False, True) in routes     # several tiles with shared queries
        if keep:
            assert all(nq > qcap for _, nq in units)


# ------------------------------------------------------------------------------------------------- D. sixteen classes
@pytest.mark.parametrize("w", [512, 1000, 8192])
@pytest.mark.parametrize("k", [15, 16])
def test_sixteen_classes(cuda, k, w):
    """K = 16 makes every one of the 32 lanes of the vertex emitter live (class c: lanes c and 16 + c)."""
    h = 48
    yt, yp = synth.layered_pair(2, h, w, k, seed=k * w, min_gap=1)
    yp[1] = synth.layered_pair(2, h, w, k, seed=k * w, min_gap=1, noise=2e-3)[1][1]
    assert all(len(np.unique(a)) == k for a in (yt[0], yp[0]))
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    longest = max(max(len(vt), len(vp)) for i in range(2) for vt, vp, _ in eo.contours(yt[i], yp[i], k, "all"))
    out = suite.contour_pass(t, p, k, mode="all", return_vertices=True, return_sq=True, max_pts=longest)
    check_contours(yt, yp, k, out, "all")
    for mode in ("all", "first"):
        check_contours(yt, yp, k, suite.contour_pass(t, p, k, mode=mode, spacing=OCT), mode, OCT)


# ------------------------------------------------------------------------------------------- E. grid-strided batches
def _small_batches(n, per):
    return [(s, min(n, s + per)) for s in range(0, n, per)]


def test_grid_strided_batches(cuda):
    """More units than SMs x 32 CTAs for components (2 N units), surface Dice (N x n_groups) and the spacing search
    (N x K x 2): every CTA handles several units in turn.  Each item equals the same item in batches that do not
    stride (no more units than SMs), and a sample with the first and the last item equals the oracle."""
    sms = torch.cuda.get_device_properties(cuda).multi_processor_count
    k, h, w = 4, 16, 32
    n = sms * MAX_BLOCKS_PER_SM + 17
    assert _groups(w, k, SD_MAX_REACH, cuda)[0] == 1
    assert 2 * n > sms * MAX_BLOCKS_PER_SM and n > sms * MAX_BLOCKS_PER_SM and n * k * 2 > sms * MAX_BLOCKS_PER_SM
    yt, yp = synth.lesion_pair(n, h, w, k, seed=5151, single_blob_interior=False)
    noisy = np.random.default_rng(5152).random(yp.shape) < 0.05
    yp[noisy] = (yp[noisy] + 1) % k
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    rng = np.random.default_rng(5153)
    sample = sorted({0, n - 1, *rng.choice(np.arange(1, n - 1), size=10, replace=False).tolist()})

    big = suite.components(t, p, k, 8)
    check_components(yt[sample], yp[sample], k, 8, big, items=sample)
    for s, e in _small_batches(n, sms // 2):
        one = suite.components(t[s:e], p[s:e], k, 8)
        assert np.array_equal(_u32(one.n_comp), _u32(big.n_comp)[s:e]) and np.array_equal(_u32(one.n_hit),
                                                                                          _u32(big.n_hit)[s:e]), s

    big = suite.surface_dice(t, p, k, PIX_TAUS)
    check_surface(yt[sample], yp[sample], k, PIX_TAUS, big, items=sample)
    for s, e in _small_batches(n, sms):
        one = suite.surface_dice(t[s:e], p[s:e], k, PIX_TAUS)
        assert np.array_equal(_u32(one.n_surf), _u32(big.n_surf)[s:e]), s
        assert np.array_equal(_u32(one.n_within), _u32(big.n_within)[s:e]), s

    for mode in ("all", "first"):
        big = suite.contour_pass(t, p, k, mode=mode, spacing=OCT)
        check_contours(yt[sample], yp[sample], k, big, mode, OCT, items=sample)
        fields = ("n_pts", "max_sq", "p95_sq", "sum_dist")
        whole = {f: getattr(big, f).cpu().numpy() for f in fields}
        for s, e in _small_batches(n, max(1, sms // (2 * k))):
            one = suite.contour_pass(t[s:e], p[s:e], k, mode=mode, spacing=OCT)
            for f in fields:
                assert np.array_equal(getattr(one, f).cpu().numpy(), whole[f][s:e]), (mode, s, f)


# ------------------------------------------------------------------------------------------- F. everything at once
def _check_result(yt, yp, k, res, taus, conn, spacing):
    ints = res.integers()
    for i in range(len(yt)):
        assert np.array_equal(ints["confusion"][i], lo.confusion_matrix(yt[i], yp[i], k)), i
    n_pts = ints["contour_n_pts"]
    for i in range(len(yt)):
        for c, (vt, vp, d) in enumerate(eo.contours(yt[i], yp[i], k, "all", spacing)):
            assert tuple(int(v) for v in n_pts[i, c]) == (len(vt), len(vp)), (i, c)
            if d is None:
                continue
            for di in (0, 1):
                vmax, lo_, hi_, s = eo.order_stats(d[di])
                assert ints["contour_max_sq"][i, c, di] == vmax, (i, c, di)
                assert tuple(ints["contour_p95_sq"][i, c, di]) == (lo_, hi_), (i, c, di)
                np.testing.assert_allclose(ints["contour_sum_dist"][i, c, di], s, rtol=1e-12, atol=0)
        ns, nw = eo.surface_counts(yt[i], yp[i], k, taus, spacing)
        assert np.array_equal(ints["surface_dice_n_surf"][i], ns) and np.array_equal(ints["surface_dice_n_within"][i], nw)
        nc, nh = eo.component_counts(yt[i], yp[i], k, conn)
        assert np.array_equal(ints["component_count"][i], nc) and np.array_equal(ints["component_hits"][i], nh)


@pytest.mark.parametrize("h,w,k", [(16, 8192, 16), (8192, 16, 3)])
def test_every_option_at_once(cuda, h, w, k):
    yt, yp = synth.layered_pair(2, h, w, k, seed=h * 3 + w + k, noise=2e-3, min_gap=1)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    for spacing, taus in ((None, (1.0, 8.0)), (OCT, (OCT[0], derive.surface_dice_spacing_limit(OCT)))):
        res = suite.evaluate(t, p, k, contours="all", surface_dice=taus, components=8, spacing=spacing)
        _check_result(yt, yp, k, res, taus, 8, spacing)
        ints, m = res.integers(), res.metrics()
        alone = [suite.evaluate(t, p, k, contours="all", spacing=spacing),
                 suite.evaluate(t, p, k, contours=False, surface_dice=taus, spacing=spacing),
                 suite.evaluate(t, p, k, contours=False, components=8, spacing=spacing)]
        for one in alone:
            for key, v in one.integers().items():
                assert np.array_equal(ints[key], v), key
            for name, v in one.metrics().items():
                assert np.array_equal(m[name], v, equal_nan=True), name


# ------------------------------------------------------------------------------------------------------ G. refusal
@pytest.mark.parametrize("h,w", [(8193, 16), (16, 8193)])
def test_sides_beyond_8192_are_refused(cuda, h, w):
    yt, yp = synth.layered_pair(1, h, w, 3, seed=h + 1)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    calls = {
        "surface_dice": lambda: suite.surface_dice(t, p, 3, (1.0,)).n_surf.cpu(),
        "surface_dice spacing": lambda: suite.surface_dice(t, p, 3, (0.01,), spacing=OCT).n_surf.cpu(),
        "components 4": lambda: suite.components(t, p, 3, 4).n_comp.cpu(),
        "components 8": lambda: suite.components(t, p, 3, 8).n_comp.cpu(),
        "contour_pass all": lambda: suite.contour_pass(t, p, 3, mode="all").max_sq.cpu(),
        "contour_pass spacing all": lambda: suite.contour_pass(t, p, 3, mode="all", spacing=OCT).max_sq.cpu(),
        "contour_pass spacing first": lambda: suite.contour_pass(t, p, 3, spacing=OCT).max_sq.cpu(),
        "evaluate all": lambda: suite.evaluate(t, p, 3, contours="all").metrics(),
        "evaluate surface_dice": lambda: suite.evaluate(t, p, 3, contours=False, surface_dice=1.0).metrics(),
        "evaluate surface_dice spacing": lambda: suite.evaluate(t, p, 3, contours=False, surface_dice=0.01,
                                                                spacing=OCT).metrics(),
        "evaluate components": lambda: suite.evaluate(t, p, 3, contours=False, components=8).metrics(),
        "evaluate spacing": lambda: suite.evaluate(t, p, 3, spacing=OCT).metrics(),
        "evaluate spacing all": lambda: suite.evaluate(t, p, 3, contours="all", spacing=OCT).metrics(),
    }
    for name, fn in calls.items():
        with pytest.raises(_lib.OctmError, match="8192"):
            fn()
            pytest.fail(f"{name} returned a result")


# ------------------------------------------------------------------------------------ packed host transfer fallback
def _wide_label_inputs(bad):
    yt, yp = synth.layered_pair(6, 48, 64, 8, seed=6100 + bad, noise=0.01)
    yp[3, 10, 20] = bad               # chunk 1 of 3 (two items per chunk), both in the AVX2 body ...
    yt[3, 47, 63] = bad               # ... and in the last label of the item
    return yt, yp


@pytest.mark.parametrize("bad", [16, 255])
def test_packed_transfer_never_changes_a_result(cuda, bad):
    """A label >= 16 has no 4-bit code: pack=True sends that chunk as it is, and the outcome is pack=False's, the same
    ValueError with validate=True and the same numbers (the pixel dropped) with validate=False."""
    yt, yp = _wide_label_inputs(bad)
    kw = dict(chunk_items=2)
    errors = []
    for pack in (False, True):
        with pytest.raises(ValueError) as e:
            suite.evaluate_host(yt, yp, 8, pack=pack, **kw).metrics()
        errors.append(str(e.value))
    assert errors[0] == errors[1]
    for opts in ({}, dict(contours="all"), dict(surface_dice=(1.0, 8.0)), dict(components=8),
                 dict(spacing=OCT, contours="all", surface_dice=0.01)):
        runs = []
        for pack in (False, True):
            res, kernels = _profiled(lambda: suite.evaluate_host(yt, yp, 8, pack=pack, validate=False, **kw, **opts))
            runs.append((res.integers(), res.metrics(), kernels))
        (ia, ma, _), (ib, mb, kb) = runs
        assert kb["unpack_nibbles_kernel"][0] == 2 * 2          # chunks 0 and 2 were packed, chunk 1 was not
        for key in ia:
            assert np.array_equal(ia[key], ib[key]), (opts, key)
        for name in ma:
            assert np.array_equal(ma[name], mb[name], equal_nan=True), (opts, name)
    clean = synth.layered_pair(6, 48, 64, 8, seed=6100 + bad, noise=0.01)
    _, kernels = _profiled(lambda: suite.evaluate_host(*clean, 8, pack=True, **kw).metrics())
    assert kernels["unpack_nibbles_kernel"][0] == 3 * 2
