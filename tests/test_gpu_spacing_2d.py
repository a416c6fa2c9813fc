"""GPU: B-scan metrics with a physical pixel spacing (``evaluate(spacing=...)``, ``contour_pass(spacing=...)``,
``surface_dice(spacing=...)``) against the pixel path at spacing (1, 1) and against ``tests/spacing_2d_oracle.py``.

Every case asserts on its inputs that it reaches the route it names: the spacing search is
``distance_spacing_kernel`` (the layered fast path and the counting search do not run), the surface Dice kernel reads
the maps byte-wise when W % 16 != 0 or a map is misaligned, and a small ``max_pts`` overflows before the retry."""
import numpy as np
import pytest

import spacing_2d_oracle as so
from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

pytestmark = pytest.mark.gpu
OCT = (0.0039, 0.0117)                      # mm: axial (rows), lateral (columns)
SPACINGS = {"oct": OCT, "rows30": (30.0, 1.0), "cols30": (1.0, 30.0), "dyadic": (0.5, 2.0)}
MODES = {"all": "all", "first": True}


def _dev(cuda, *arrs):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).to(cuda) for a in arrs)


def _profiled(fn):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    with _lib.kernel_profile() as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, prof.kernels


def _inputs(case, cuda):
    if case == "cfg4_clean":
        return (*synth.layered_pair_device(6, 496, 512, 8, seed=4004, device=cuda), 8)
    if case == "cfg4_noise":
        return (*synth.layered_pair_device(6, 496, 512, 8, seed=4004, device=cuda, noise=0.002), 8)
    if case == "ragged":
        return (*synth.ragged_pair_device(6, 496, 512, 8, seed=9, device=cuda), 8)
    yt, yp = synth.lesion_pair(6, 256, 256, 4, seed=3, single_blob_interior=False)
    return (*_dev(cuda, yt, yp), 4)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("case", ["cfg4_clean", "cfg4_noise", "ragged", "lesion"])
def test_unit_spacing_is_the_pixel_path(cuda, case, mode):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp, k = _inputs(case, cuda)
    px = suite.evaluate(yt, yp, k, contours=MODES[mode], surface_dice=(1.0, 2.0, 8.0), boundaries=True)
    sp, kernels = _profiled(lambda: suite.evaluate(yt, yp, k, contours=MODES[mode], surface_dice=(1.0, 2.0, 8.0),
                                                   boundaries=True, spacing=(1, 1)))
    assert "distance_spacing_kernel" in kernels
    assert not any(name.startswith(("layered_distance", "distance_column", "distance_select")) for name in kernels)
    ia, ib = px.integers(), sp.integers()
    assert ib["contour_max_sq"].dtype == ib["contour_p95_sq"].dtype == np.float64
    for key in ("contour_max_sq", "contour_p95_sq"):
        assert np.array_equal(ib[key], ia[key].astype(np.float64)), key
    for key in ("contour_n_pts", "surface_dice_n_surf", "surface_dice_n_within", "confusion", "thickness_absdiff"):
        assert np.array_equal(ib[key], ia[key]), key
    ma, mb = px.metrics(), sp.metrics()
    for name in ("hausdorff_distance", "hausdorff_distance_95", "thickness_difference", "boundary_mse", "boundary_rmse",
                 "boundary_mad", "surface_dice", "dice_coefficient"):
        assert np.array_equal(mb[name], ma[name], equal_nan=True), name
    assert np.array_equal(np.isnan(mb["assd"]), np.isnan(ma["assd"]))
    np.testing.assert_allclose(mb["assd"], ma["assd"], rtol=1e-12, atol=0)
    host = sp.metrics_host()                   # derive.py mirrors the device epilogue bit for bit
    for name in host:
        assert np.array_equal(host[name], mb[name], equal_nan=True), name
    # every stored d2 (same vertices, same slots) equals the pixel D2
    a = suite.contour_pass(yt, yp, k, return_vertices=True, return_sq=True, mode="all" if mode == "all" else "first")
    b = suite.contour_pass(yt, yp, k, return_vertices=True, return_sq=True, mode="all" if mode == "all" else "first",
                           spacing=(1.0, 1.0))
    n_pts = a.n_pts.cpu().numpy().view(np.uint32)
    assert np.array_equal(b.n_pts.cpu().numpy().view(np.uint32), n_pts)
    va, vb = a.verts.cpu().numpy(), b.verts.cpu().numpy()
    sa, sb = a.sq.cpu().numpy().view(np.uint32), b.sq.cpu().numpy()
    for i in range(n_pts.shape[0]):
        for c in range(k):
            for side in range(2):
                m = min(int(n_pts[i, c, side]), va.shape[-1])
                assert np.array_equal(vb[i, c, side, :m], va[i, c, side, :m]), (i, c, side)
            if n_pts[i, c, 0] == 0 or n_pts[i, c, 1] == 0:
                continue
            for d in range(2):
                m = int(n_pts[i, c, 1 - d])
                assert np.array_equal(sb[i, c, d, :m], sa[i, c, d, :m].astype(np.float64)), (i, c, d)


def _oracle_inputs(cuda):
    yt, yp = synth.layered_pair(3, 40, 64, 5, seed=21, noise=0.02)
    yield "layered", yt, yp, 5
    yt, yp = synth.lesion_pair(3, 48, 56, 3, seed=22, single_blob_interior=False)
    yield "lesion", yt, yp, 3
    rng = np.random.default_rng(23)
    yield "random", (rng.random((3, 17, 23)) < 0.4).astype(np.uint8), (rng.random((3, 17, 23)) < 0.5).astype(np.uint8), 2


def _check_against_oracle(out, yt, yp, k, spacing, mode):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    n_pts = out.n_pts.cpu().numpy().view(np.uint32)
    verts, sq = out.verts.cpu().numpy().view(np.uint32), out.sq.cpu().numpy()
    max_sq, p95, sums = out.max_sq.cpu().numpy(), out.p95_sq.cpu().numpy(), out.sum_dist.cpu().numpy()
    m = derive.contour_metrics(n_pts, max_sq, p95, sums)
    seen = 0
    for i in range(yt.shape[0]):
        for c in range(k):
            vt, vp = so.vertices(yt[i] == c, mode), so.vertices(yp[i] == c, mode)
            if vt is None or vp is None:
                assert np.isnan(m["hausdorff_distance"][i, c]), (i, c)
                continue
            seen += 1
            got = []
            for side, ref in ((0, vt), (1, vp)):
                v = verts[i, c, side, :n_pts[i, c, side]]
                g = np.stack([v >> 16, v & 0xffff], axis=1).astype(np.int64)
                assert sorted(map(tuple, g)) == sorted(map(tuple, ref)), (i, c, side)     # the oracle's vertex multiset
                got.append(g)
            ds = []
            for d, (src, qry) in enumerate(((got[0], got[1]), (got[1], got[0]))):
                want = so.squared_distances(src, qry, spacing)
                assert np.array_equal(sq[i, c, d, :len(qry)], want), (i, c, d)
                assert (max_sq[i, c, d], p95[i, c, d, 0], p95[i, c, d, 1]) == so.order_statistics(want), (i, c, d)
                ds.append(want)
            ref = lo.contour_metrics_from_sq(ds[0], ds[1])
            assert m["hausdorff_distance"][i, c] == ref["hausdorff_distance"]
            np.testing.assert_allclose(m["assd"][i, c], ref["assd"], rtol=1e-12, atol=0)
            np.testing.assert_allclose(m["hausdorff_distance_95"][i, c], ref["hausdorff_distance_95"], rtol=1e-12, atol=0)
    return seen


@pytest.mark.parametrize("mode", ["all", "first"])
@pytest.mark.parametrize("spacing", list(SPACINGS))
def test_against_the_oracle(cuda, spacing, mode):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    seen = 0
    for _, yt, yp, k in _oracle_inputs(cuda):
        dt, dp = _dev(cuda, yt, yp)
        out, kernels = _profiled(lambda: suite.contour_pass(dt, dp, k, return_vertices=True, return_sq=True, mode=mode,
                                                            spacing=SPACINGS[spacing], max_pts=1024))
        assert "distance_spacing_kernel" in kernels
        seen += _check_against_oracle(out, yt, yp, k, SPACINGS[spacing], mode)
    assert seen >= 15


def _nsd_check(yt, yp, k, spacing, taus, res):
    ints = res.integers()
    for i in range(yt.shape[0]):
        for c in range(k):
            n_surf, n_within = so.surface_dice_counts(yt[i] == c, yp[i] == c, spacing, taus)
            assert tuple(ints["surface_dice_n_surf"][i, c]) == n_surf, (i, c)
            assert np.array_equal(ints["surface_dice_n_within"][i, c], n_within), (i, c)


@pytest.mark.parametrize("spacing", list(SPACINGS))
def test_surface_dice_against_the_oracle(cuda, spacing):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, suite
    sp = SPACINGS[spacing]
    lim = derive.surface_dice_spacing_limit(sp)
    taus = (0.0, lim / 4, lim / 2, lim)
    for _, yt, yp, k in _oracle_inputs(cuda):
        res = suite.evaluate(*_dev(cuda, yt, yp), k, contours=False, surface_dice=taus, spacing=sp)
        _nsd_check(yt, yp, k, sp, taus, res)


def test_surface_dice_tolerance_ties(cuda):
    """Dyadic spacing: every q is exact, so a tolerance equal to a distance that occurs counts that vertex; so do the
    largest tolerances allowed when the rows bound the reach and when the columns do."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, suite
    _, yt, yp, k = next(iter(_oracle_inputs(cuda)))
    for sp in ((0.5, 2.0), (2.0, 0.5)):
        occurring = np.unique(np.concatenate([so.intermediates(yt[i] == c, yp[i] == c, sp)["sq_pred_to_true"]
                                              for i in range(yt.shape[0]) for c in range(k)
                                              if so.intermediates(yt[i] == c, yp[i] == c, sp) is not None]))
        dist = np.sqrt(occurring / 4.0)
        lim = derive.surface_dice_spacing_limit(sp)
        ties = tuple(float(x) for x in dist[(dist > 0) & (dist <= lim)][:2]) + (lim, 0.0)
        res = suite.evaluate(*_dev(cuda, yt, yp), k, contours=False, surface_dice=ties, spacing=sp)
        _nsd_check(yt, yp, k, sp, ties, res)
        with pytest.raises(ValueError, match="largest tolerance"):
            suite.evaluate(*_dev(cuda, yt, yp), k, contours=False, surface_dice=float(np.nextafter(lim, 99)), spacing=sp)


def test_byte_wise_loader(cuda):
    """W % 16 != 0 and misaligned maps take the surface Dice kernel's byte-wise loads."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = synth.lesion_pair(3, 40, 60, 3, seed=31, single_blob_interior=False)
    assert yt.shape[2] % 16 != 0
    taus = (0.004, 0.02)
    _nsd_check(yt, yp, 3, OCT, taus, suite.evaluate(*_dev(cuda, yt, yp), 3, contours="all", surface_dice=taus,
                                                    spacing=OCT))
    yt, yp = synth.lesion_pair(3, 32, 64, 3, seed=32, single_blob_interior=False)
    bufs = [torch.empty(a.size + 1, dtype=torch.uint8, device=cuda) for a in (yt, yp)]
    views = [b[1:].view(a.shape).copy_(torch.from_numpy(a)) for a, b in zip((yt, yp), bufs)]
    assert all(v.is_contiguous() and v.data_ptr() % 16 == 1 for v in views)
    _nsd_check(yt, yp, 3, OCT, taus, suite.evaluate(*views, 3, contours=True, surface_dice=taus, spacing=OCT))


@pytest.mark.parametrize("mode", list(MODES))
def test_overflow_retry(cuda, mode):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    yt, yp = _dev(cuda, *synth.layered_pair(5, 64, 96, 6, seed=41, noise=0.01))
    first = suite.contour_pass(yt, yp, 6, max_pts=16, check_overflow=False, mode="all" if mode == "all" else "first",
                               spacing=OCT)
    assert bool(((first.flags & (_lib.CF_TRUE_OVERFLOW | _lib.CF_PRED_OVERFLOW)) != 0).any())
    small = suite.evaluate(yt, yp, 6, contours=MODES[mode], max_pts=16, spacing=OCT)
    big = suite.evaluate(yt, yp, 6, contours=MODES[mode], max_pts=8192, spacing=OCT)
    a, b = small.integers(), big.integers()
    for key in ("contour_n_pts", "contour_max_sq", "contour_p95_sq", "contour_sum_dist"):
        assert np.array_equal(a[key], b[key]), key
    for name, v in big.metrics().items():
        assert np.array_equal(small.metrics()[name], v, equal_nan=True), name


def test_empty_boundaries(cuda):
    """A class absent from both maps: NaN distances, NSD NaN; absent from one map only: NaN distances, NSD 0."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt = np.zeros((2, 16, 20), np.uint8)
    yp = np.zeros((2, 16, 20), np.uint8)
    yt[:, 4:9, 5:12] = 1                        # class 1 in y_true only; class 2 nowhere
    for mode in MODES.values():
        res = suite.evaluate(*_dev(cuda, yt, yp), 3, contours=mode, surface_dice=(0.01,), spacing=OCT)
        m = res.metrics()
        assert np.isnan(m["hausdorff_distance"][:, 1:]).all() and np.isnan(m["assd"][:, 1:]).all()
        assert (m["surface_dice"][:, 1, 0] == 0).all() and np.isnan(m["surface_dice"][:, 2, 0]).all()


def test_evaluate_host_chunks_and_dataset_totals(cuda):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist, suite
    yt, yp = synth.layered_pair(7, 48, 64, 5, seed=51, noise=0.01)
    whole = suite.evaluate(*_dev(cuda, yt, yp), 5, contours="all", surface_dice=(0.01,), spacing=OCT)
    parts = suite.evaluate_host(yt, yp, 5, contours="all", surface_dice=(0.01,), spacing=OCT, chunk_items=3)
    assert parts.spacing == whole.spacing == OCT
    a, b = whole.integers(), parts.integers()
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    ma, mb = whole.metrics(), parts.metrics()
    for name in ma:
        assert np.array_equal(ma[name], mb[name], equal_nan=True), name
    tot = dist.dataset_totals(whole, 1)
    plain = dist.unpack(whole.totals_host()[:dist.base_len(5)], 5, 64)
    assert np.array_equal(tot["thickness_difference"], plain["thickness_difference"] * OCT[0])
    assert np.array_equal(tot["boundary_mad"], plain["boundary_mad"] * OCT[0])


def test_repeat_determinism(cuda):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp, k = _inputs("ragged", cuda)
    runs = [suite.evaluate(yt, yp, k, contours="all", surface_dice=(0.004, 0.01), spacing=OCT).integers()
            for _ in range(3)]
    for key in runs[0]:
        for r in runs[1:]:
            assert np.array_equal(r[key], runs[0][key]), key
