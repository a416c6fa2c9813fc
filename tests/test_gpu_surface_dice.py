"""GPU: normalized surface Dice counts (octm_surface_dice_u8, evaluate(surface_dice=...)) equal the oracle exactly."""
import numpy as np
import pytest

from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, synth
import surface_dice_oracle as so_

pytestmark = pytest.mark.gpu

EDGE_TAUS = (0.0, np.sqrt(2) / 2, 1.0, np.sqrt(5) / 2, 8.0)
TAU_SETS = [EDGE_TAUS[:4], (8.0, np.nextafter(np.sqrt(2) / 2, -np.inf), np.nextafter(1.0, -np.inf), 2.0),
            (np.nextafter(8.0, -np.inf), 3.0, 0.5, np.nextafter(np.sqrt(5) / 2, -np.inf))]


def _dev(a, cuda):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _counts(t, p, k, taus):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    out = suite.surface_dice(t, p, k, taus)
    torch.cuda.synchronize()
    assert out.tolerances == tuple(float(x) for x in taus)
    return out.n_surf.cpu().numpy().view(np.uint32), out.n_within.cpu().numpy().view(np.uint32)


def _check(yt, yp, k, taus, cuda, t=None, p=None):
    t = _dev(yt, cuda) if t is None else t
    p = _dev(yp, cuda) if p is None else p
    ns, nw = _counts(t, p, k, taus)
    ref_ns, ref_nw = so_.label_counts(yt, yp, k, taus)
    np.testing.assert_array_equal(ns, ref_ns)
    np.testing.assert_array_equal(nw, ref_nw)
    return nw


def test_random_binary_masks(cuda):
    """1 x 1 to 20 x 20: holes, an absent class, a class filling the map, identical maps."""
    rng = np.random.default_rng(101)
    for it in range(24):
        h, w = (1, 1) if it == 0 else rng.integers(1, 21, size=2)
        n = 6
        a = (rng.random((n, h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8)
        b = (rng.random((n, h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8)
        a[0] = 0
        b[1] = 1
        a[2] = b[2]
        yy, xx = np.ogrid[:h, :w]
        a[3] = ((yy - h / 2) ** 2 + (xx - w / 2) ** 2 < (min(h, w) / 3) ** 2)
        a[3][h // 2, w // 2] = 0                          # a hole
        for taus in TAU_SETS:
            _check(a, b, 2, taus, cuda)


def _offsets(d2):
    r = int(np.ceil(np.sqrt(d2)))
    return [(dy, dx) for dy in range(-r, r + 1) for dx in range(-r, r + 1)
            if dy * dy + dx * dx == d2 and (dy - dx) % 2 == 0]


def test_hand_made_offsets_at_segment_band_and_image_edges(cuda):
    """A one-pixel blob in each map, placed so that some vertex pair lies at lattice offset (dy, dx) exactly, for every
    offset of D2 in {2, 4, 8, 10, 16, 250, 256, 260} (254 and 258 are no vertex offset: every D2 of two vertices is
    0 or 2 mod 4 with dy == dx (mod 2)), around the corners, the 512-column segment edges and the 8-row band edges."""
    h, w = 34, 1100
    assert not _offsets(254) and not _offsets(258)
    anchors = [(0, 0), (h - 1, w - 1), (0, w - 1), (h - 1, 0)]
    anchors += [(y, x) for y in (7, 8, 15, 16, 23, 24) for x in (3, 511, 512, 1023, 1024)]
    items = []
    for d2 in (2, 4, 8, 10, 16, 250, 256, 260):
        for dy, dx in _offsets(d2):
            # single pixels at pixel offset (oy, ox): their crack diamonds hold a vertex pair at (dy, dx) exactly
            oy, ox = (dy // 2, dx // 2) if dy % 2 == 0 else ((dy - 1) // 2, (dx - 1) // 2)
            for y, x in anchors:
                if 0 <= y + oy < h and 0 <= x + ox < w:
                    items.append((y, x, y + oy, x + ox))
    yt = np.zeros((len(items), h, w), np.uint8)
    yp = np.zeros_like(yt)
    for i, (y, x, y1, x1) in enumerate(items):
        yt[i, y, x] = 1
        yp[i, y1, x1] = 1
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    for d2s in ((2, 4, 8, 10), (16, 250, 254, 256)):
        taus = tuple(np.sqrt(d / 4.0) for d in d2s)
        below = tuple(np.nextafter(x, -np.inf) for x in taus)
        assert [derive.surface_dice_threshold(x) for x in taus] == list(d2s)
        ref_ns, ref_nw = so_.label_counts(yt, yp, 2, taus + below)
        for j, ts in enumerate((taus, below)):
            ns, nw = _counts(t, p, 2, ts)
            np.testing.assert_array_equal(ns, ref_ns)
            np.testing.assert_array_equal(nw, ref_nw[..., 4 * j:4 * j + 4], err_msg=str(ts))


@pytest.mark.parametrize("case", ["layered6", "layered8_noise", "lesion_multi", "k10_w1000", "k16", "k16_w2048",
                                  "odd_unaligned"])
def test_multiclass(cuda, case):
    taus = (1.0, 2.0, np.sqrt(5) / 2, 8.0)
    if case == "layered6":
        yt, yp, k = *synth.layered_pair(3, 64, 128, 6, seed=111), 6
    elif case == "layered8_noise":
        yt, yp, k = *synth.layered_pair(3, 96, 160, 8, seed=112, noise=0.01), 8
    elif case == "lesion_multi":
        yt, yp, k = *synth.lesion_pair(3, 96, 128, 4, seed=113, single_blob_interior=False), 4
    elif case == "k10_w1000":
        yt, yp, k = *synth.layered_pair(2, 64, 1000, 10, seed=114, noise=0.002), 10      # two 512-column segments
    elif case == "k16":
        yt, yp, k = *synth.layered_pair(2, 80, 96, 16, seed=115, noise=0.01, min_gap=1), 16
    elif case == "k16_w2048":        # at tau = 8 the ring of 16 classes exceeds shared memory: two class groups
        yt, yp, k = *synth.layered_pair(2, 40, 2048, 16, seed=117, noise=0.005, min_gap=1), 16
    else:
        rng = np.random.default_rng(116)
        yt = rng.integers(0, 5, size=(4, 33, 50), dtype=np.uint8)
        yp = yt.copy()
        yp[rng.random(yp.shape) < 0.2] = 2
        t, p = _dev(yt, cuda)[1:], _dev(yp, cuda)[1:]      # items start 1650 B into the allocation: byte loader
        assert t.data_ptr() % 16 != 0
        _check(yt[1:], yp[1:], 5, taus, cuda, t, p)
        _check(yt[1:], yp[1:], 5, (0.5, 3.0), cuda, t, p)
        return
    _check(yt, yp, k, taus, cuda)


def _full_size_pairs(cuda):
    import torch
    n = 3
    yield "clean", synth.layered_pair_device(n, 496, 512, 8, seed=4004, device=cuda)
    yield "noise", synth.layered_pair_device(n, 496, 512, 8, seed=4004, device=cuda, noise=0.002)
    yield "ragged", synth.ragged_pair_device(n, 496, 512, 8, seed=4005, device=cuda)
    g = torch.Generator(device=cuda).manual_seed(4006)
    yield "uniform", tuple(torch.randint(0, 8, (2, 496, 512), generator=g, device=cuda, dtype=torch.uint8) for _ in range(2))


def test_full_size_against_all_contour_distances(cuda):
    """cfg4-size items: n_surf is the all-contour n_pts and n_within counts the stored squared distances <= T_j."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    taus = (1.0, np.sqrt(5) / 2, 2.0, 8.0)
    thr = np.array([derive.surface_dice_threshold(x) for x in taus])
    for name, (t, p) in _full_size_pairs(cuda):
        ns, nw = _counts(t, p, 8, taus)
        probe = suite.contour_pass(t, p, 8, mode="all", max_pts=8, check_overflow=False)     # exact counts
        torch.cuda.synchronize()
        need = (int(probe.n_pts.max()) + 3) & ~3
        ct = suite.contour_pass(t, p, 8, mode="all", return_sq=True, max_pts=max(need, 8))
        torch.cuda.synchronize()
        n_pts = ct.n_pts.cpu().numpy().view(np.uint32)
        sq = ct.sq.cpu().numpy().view(np.uint32)
        np.testing.assert_array_equal(ns, n_pts, err_msg=name)
        for i, c, d in np.ndindex(ns.shape[0], 8, 2):
            m = n_pts[i, c, 1 - d]                  # direction 0 queries the pred vertices
            if n_pts[i, c, d] == 0:
                want = np.zeros(len(taus), np.int64)
            else:
                want = (sq[i, c, d, :m][:, None] <= thr[None, :]).sum(0)
            np.testing.assert_array_equal(nw[i, c, d], want, err_msg=f"{name} {i} {c} {d}")
        del ct, sq


def test_suite_integration(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist, suite
    yt, yp = synth.layered_pair(12, 64, 128, 6, seed=121, noise=0.01)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    res = suite.evaluate(t, p, 6, surface_dice=(2.0, 1.0))
    assert res.surface_dice_tolerances == (2.0, 1.0)
    m, mh = res.metrics(), res.metrics_host()
    assert m["surface_dice"].shape == (12, 6, 2) and m["surface_dice"].dtype == np.float64
    for key in mh:
        np.testing.assert_array_equal(m[key], mh[key], err_msg=key)
    ref_ns, ref_nw = so_.label_counts(yt, yp, 6, (2.0, 1.0))          # the caller's order
    ints = res.integers()
    np.testing.assert_array_equal(ints["surface_dice_n_surf"], ref_ns)
    np.testing.assert_array_equal(ints["surface_dice_n_within"], ref_nw)
    np.testing.assert_array_equal(m["surface_dice"], derive.surface_dice(ref_ns, ref_nw))
    # everything else is what evaluate() gives without it
    base = suite.evaluate(t, p, 6)
    assert base.surface_dice_tolerances is None and "surface_dice" not in base.metrics()
    assert set(m) - set(base.metrics()) == {"surface_dice"}
    for key, v in base.metrics().items():
        np.testing.assert_array_equal(m[key], v, err_msg=key)
    bi = base.integers()
    assert set(ints) - set(bi) == {"surface_dice_n_surf", "surface_dice_n_within"}
    for key, v in bi.items():
        assert np.array_equal(ints[key].view(np.uint8), v.view(np.uint8)), key
    np.testing.assert_array_equal(res.totals_host(), base.totals_host())
    # the surface is the whole boundary whatever the contour mode
    for contours in (True, "all", False):
        other = suite.evaluate(t, p, 6, contours=contours, surface_dice=(2.0, 1.0)).metrics()
        np.testing.assert_array_equal(other["surface_dice"], m["surface_dice"], err_msg=str(contours))
    host = suite.evaluate_host(yt, yp, 6, chunk_items=5, surface_dice=(2.0, 1.0))
    assert host.surface_dice_tolerances == (2.0, 1.0)
    for key, v in m.items():
        np.testing.assert_array_equal(host.metrics()[key], v, err_msg=key)
    for key, v in ints.items():
        np.testing.assert_array_equal(host.integers()[key], v, err_msg=key)
    tot = dist.surface_dice_totals(res, 1)
    nsd = m["surface_dice"]
    np.testing.assert_array_equal(tot["surface_dice_items"], (~np.isnan(nsd)).sum(0))
    np.testing.assert_allclose(tot["surface_dice_mean"], np.nanmean(nsd, axis=0), rtol=1e-12)
    empty = suite.evaluate(t[:0], p[:0], 6, surface_dice=(1.0, 2.0, 3.0))
    assert empty.metrics()["surface_dice"].shape == (0, 6, 3)
    for bad in (9.0, -1.0, float("nan"), (), (1.0, 2.0, 3.0, 4.0, 5.0)):
        with pytest.raises(ValueError):
            suite.evaluate(t, p, 6, surface_dice=bad)
        with pytest.raises(ValueError):
            suite.surface_dice(t, p, 6, bad)
    torch.cuda.synchronize()


def test_kernel_launches(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, _lib
    yt, yp = synth.lesion_pair(4, 96, 128, 4, seed=131, single_blob_interior=False)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    with _lib.kernel_profile() as prof:
        suite.evaluate(t, p, 4).metrics()
        torch.cuda.synchronize()
    assert "surface_dice_kernel" not in prof.kernels
    with _lib.kernel_profile() as prof:
        suite.evaluate(t, p, 4, surface_dice=(1.0, 2.0)).metrics()
        torch.cuda.synchronize()
    assert prof.kernels["surface_dice_kernel"][0] == 1
    with _lib.kernel_profile() as prof:
        suite.evaluate_host(yt, yp, 4, chunk_items=2, surface_dice=1.0).metrics()
        torch.cuda.synchronize()
    assert prof.kernels["surface_dice_kernel"][0] == 2             # one launch per chunk
