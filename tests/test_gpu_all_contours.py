"""GPU: all-contour vertices, exact squared distances and hausdorff / hd95 / assd (contours="all") vs the oracle."""
import numpy as np
import pytest

from oracle import contours_oracle as co
from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import synth
import all_contours_oracle as ao

pytestmark = pytest.mark.gpu
RTOL = 1e-6


def _dev(a, cuda):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _all_pass(yt, yp, k, **kw):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    out = suite.contour_pass(yt, yp, k, return_vertices=True, return_sq=True, mode="all", **kw)
    torch.cuda.synchronize()
    return out


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _check(yt, yp, k, out):
    """Every (item, class): stored vertices, counts and per-query squared distances equal the oracle's exactly."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    n_pts, verts, sq = _u32(out.n_pts), _u32(out.verts), _u32(out.sq)
    flags = _u32(out.flags)
    assert not (flags & 3).any()                       # *_CLOSED never set in this mode
    m = derive.contour_metrics(n_pts, _u32(out.max_sq), _u32(out.p95_sq), out.sum_dist.cpu().numpy())
    for i in range(yt.shape[0]):
        for c in range(k):
            vt, vp = ao.all_vertices(yt[i] == c), ao.all_vertices(yp[i] == c)
            assert n_pts[i, c, 0] == len(vt) and n_pts[i, c, 1] == len(vp), (i, c)
            np.testing.assert_array_equal(verts[i, c, 0, :len(vt)], ao.pack(vt), err_msg=f"true {i} {c}")
            np.testing.assert_array_equal(verts[i, c, 1, :len(vp)], ao.pack(vp), err_msg=f"pred {i} {c}")
            im = ao.all_contour_intermediates(yt[i] == c, yp[i] == c)
            if im is None:
                assert np.isnan(m["hausdorff_distance"][i, c])
                continue
            np.testing.assert_array_equal(sq[i, c, 0, :len(vp)], im["sq_pred_to_true"], err_msg=f"d0 {i} {c}")
            np.testing.assert_array_equal(sq[i, c, 1, :len(vt)], im["sq_true_to_pred"], err_msg=f"d1 {i} {c}")
            ref = lo.contour_metrics_from_sq(im["sq_pred_to_true"], im["sq_true_to_pred"])
            assert m["hausdorff_distance"][i, c] == ref["hausdorff_distance"], (i, c)
            for name in ("hausdorff_distance_95", "assd"):
                np.testing.assert_allclose(m[name][i, c], ref[name], rtol=RTOL, atol=0, err_msg=f"{name} {i} {c}")
    return m


def test_random_binary_masks(cuda):
    """Saddles, holes, border-touching shapes, absent classes, masks that fill the image."""
    rng = np.random.default_rng(77)
    for _ in range(30):
        h, w = rng.integers(2, 21, size=2)
        n = 6
        a = (rng.random((n, h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8)
        b = (rng.random((n, h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8)
        a[0] = 0
        b[1] = 1
        a[2] = b[2]
        yy, xx = np.ogrid[:h, :w]
        a[3] = ((yy - h / 2) ** 2 + (xx - w / 2) ** 2 < (min(h, w) / 3) ** 2)
        a[3][h // 2, w // 2] = 0                         # a hole: two closed contours
        _check(a, b, 2, _all_pass(_dev(a, cuda), _dev(b, cuda), 2, max_pts=2048))


@pytest.mark.parametrize("case", ["layered6", "layered8_noise", "lesion_single", "lesion_multi", "k10_wide", "odd_unaligned"])
def test_multiclass(cuda, case):
    if case == "layered6":
        yt, yp, k = *synth.layered_pair(3, 64, 128, 6, seed=11), 6
    elif case == "layered8_noise":
        yt, yp, k = *synth.layered_pair(3, 96, 160, 8, seed=12, noise=0.01), 8
    elif case == "lesion_single":
        yt, yp, k = *synth.lesion_pair(3, 96, 128, 4, seed=13, single_blob_interior=True), 4
    elif case == "lesion_multi":
        yt, yp, k = *synth.lesion_pair(3, 96, 128, 4, seed=14, single_blob_interior=False), 4
    elif case == "k10_wide":
        yt, yp, k = *synth.layered_pair(2, 96, 1000, 10, seed=15, noise=0.002), 10     # two 512-column segments
    else:
        rng = np.random.default_rng(16)
        yt = rng.integers(0, 5, size=(4, 33, 50), dtype=np.uint8)
        yp = yt.copy()
        yp[rng.random(yp.shape) < 0.2] = 2
        k = 5
    if case == "odd_unaligned":
        import torch
        t, p = _dev(yt, cuda), _dev(yp, cuda)
        out = _all_pass(t[1:], p[1:], k)                 # items start 1650 B into the allocation: not 16-byte aligned
        assert t[1:].data_ptr() % 16 != 0
        _check(yt[1:], yp[1:], k, out)
        torch.cuda.synchronize()
        return
    _check(yt, yp, k, _all_pass(_dev(yt, cuda), _dev(yp, cuda), k))


def test_sq_equals_distance_transform(cuda):
    """Independent check of D2: the EDT of the doubled lattice, whatever the oracle picks for small sets."""
    yt, yp = synth.layered_pair(2, 80, 96, 5, seed=21, noise=0.01)
    out = _all_pass(_dev(yt, cuda), _dev(yp, cuda), 5)
    n_pts, sq = _u32(out.n_pts), _u32(out.sq)
    for i in range(2):
        for c in range(5):
            vt, vp = ao.all_vertices(yt[i] == c), ao.all_vertices(yp[i] == c)
            if len(vt) == 0 or len(vp) == 0:
                continue
            np.testing.assert_array_equal(sq[i, c, 0, :n_pts[i, c, 1]], ao.edt_sq_distances(vt, vp, yt.shape[1:]))
            np.testing.assert_array_equal(sq[i, c, 1, :n_pts[i, c, 0]], ao.edt_sq_distances(vp, vt, yt.shape[1:]))


def test_relation_to_contour_zero(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, suite
    yt, yp = synth.lesion_pair(4, 96, 128, 4, seed=31, single_blob_interior=True)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    first = suite.contour_pass(t, p, 4)
    allc = suite.contour_pass(t, p, 4, mode="all")
    torch.cuda.synchronize()
    nf, na = _u32(first.n_pts), _u32(allc.n_pts)
    hf = derive.contour_metrics(nf, _u32(first.max_sq), _u32(first.p95_sq), first.sum_dist.cpu().numpy())
    ha = derive.contour_metrics(na, _u32(allc.max_sq), _u32(allc.p95_sq), allc.sum_dist.cpu().numpy())
    single = pairs = 0
    for i in range(4):
        for c in range(4):
            one = [len(co.find_contours((lab[i] == c).astype(np.uint8), 0.5)) == 1 for lab in (yt, yp)]
            for m in range(2):
                if one[m]:
                    assert na[i, c, m] == nf[i, c, m] - 1, (i, c, m)      # contour [0] repeats its closing vertex
                    single += 1
            if all(one):
                assert ha["hausdorff_distance"][i, c] == hf["hausdorff_distance"][i, c], (i, c)
                pairs += 1
            if c == 0:                                   # background: the blobs are holes, i.e. further contours
                assert na[i, 0, 0] > nf[i, 0, 0] and na[i, 0, 1] > nf[i, 0, 1]
    assert single > 0 and pairs > 0
    # a middle layer of a layered map has an upper and a lower boundary; contour [0] is the upper one only
    yt, yp = synth.layered_pair(2, 64, 128, 6, seed=32)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    nf = _u32(suite.contour_pass(t, p, 6).n_pts)
    na = _u32(suite.contour_pass(t, p, 6, mode="all").n_pts)
    assert (na[:, 3] > nf[:, 3]).all()


def test_overflow_retry_matches_a_large_bound(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, _lib
    yt, yp = synth.layered_pair(5, 64, 128, 6, seed=41, noise=0.005)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    big = suite.evaluate(t, p, 6, contours="all", max_pts=4096)
    small = suite.evaluate(t, p, 6, contours="all", max_pts=16)
    ib, is_ = big.integers(), small.integers()
    for key in ("contour_n_pts", "contour_flags", "contour_max_sq", "contour_p95_sq", "contour_sum_dist"):
        np.testing.assert_array_equal(is_[key], ib[key], err_msg=key)
    mb, ms = big.metrics(), small.metrics()
    for key in mb:
        np.testing.assert_array_equal(ms[key], mb[key], err_msg=key)
    # contour_pass retries on its own; exact counts make it one round
    cp = suite.contour_pass(t, p, 6, mode="all", max_pts=16)
    np.testing.assert_array_equal(cp.sum_dist.cpu().numpy(), ib["contour_sum_dist"])
    need = (int(_u32(big.contours.n_pts).max()) + 3) & ~3
    with pytest.raises(_lib.OctmError, match=f"max_pts >= {need}"):
        suite.contour_pass(t, p, 6, mode="all", max_pts=16, return_vertices=True)
    torch.cuda.synchronize()


def _edt_stats(yt, yp, k):
    """max_sq, the two p95 order statistics and sum_dist per (item, class, direction) from the EDT oracle."""
    n = yt.shape[0]
    mx = np.zeros((n, k, 2), np.int64)
    p95 = np.zeros((n, k, 2, 2), np.int64)
    sd = np.zeros((n, k, 2))
    for i in range(n):
        for c in range(k):
            vt, vp = ao.all_vertices(yt[i] == c), ao.all_vertices(yp[i] == c)
            for d, (src, qry) in enumerate(((vt, vp), (vp, vt))):
                s = np.sort(ao.edt_sq_distances(src, qry, yt.shape[1:]))
                lo_ = int(np.floor((len(s) - 1) * 0.95))
                mx[i, c, d] = s[-1]
                p95[i, c, d] = (s[lo_], s[min(lo_ + 1, len(s) - 1)])
                sd[i, c, d] = np.sum(np.sqrt(s / 4.0))
    return mx, p95, sd


def test_uniform_random_labels_exceed_the_first_bound_and_complete(cuda):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    rng = np.random.default_rng(51)
    yt = rng.integers(0, 8, size=(2, 496, 512), dtype=np.uint8)
    yp = rng.integers(0, 8, size=(2, 496, 512), dtype=np.uint8)
    res = suite.evaluate(_dev(yt, cuda), _dev(yp, cuda), 8, contours="all")
    ints = res.integers()
    n_pts = ints["contour_n_pts"]
    assert n_pts.min() > 65536 and n_pts.max() <= suite.crack_bound(496, 512)
    assert not (ints["contour_flags"] & 12).any()
    mx, p95, sd = _edt_stats(yt, yp, 8)
    np.testing.assert_array_equal(ints["contour_max_sq"], mx)
    np.testing.assert_array_equal(ints["contour_p95_sq"], p95)
    np.testing.assert_allclose(ints["contour_sum_dist"], sd, rtol=1e-9)


def test_two_runs_are_bit_identical(cuda):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = synth.lesion_pair(6, 128, 160, 4, seed=61, single_blob_interior=False)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    a = _all_pass(t, p, 4)
    b = _all_pass(t, p, 4)
    for f in ("n_pts", "flags", "max_sq", "p95_sq"):
        assert np.array_equal(_u32(getattr(a, f)), _u32(getattr(b, f))), f
    n_pts = _u32(a.n_pts)
    va, vb, sa, sb = _u32(a.verts), _u32(b.verts), _u32(a.sq), _u32(b.sq)
    for i, c in np.ndindex(*n_pts.shape[:2]):          # the entries past a list's count are not written
        for m in range(2):
            assert np.array_equal(va[i, c, m, :n_pts[i, c, m]], vb[i, c, m, :n_pts[i, c, m]]), (i, c, m)
            assert np.array_equal(sa[i, c, m, :n_pts[i, c, 1 - m]], sb[i, c, m, :n_pts[i, c, 1 - m]]), (i, c, m)
    assert np.array_equal(a.sum_dist.cpu().numpy().view(np.uint64), b.sum_dist.cpu().numpy().view(np.uint64))
    ra = suite.evaluate(t, p, 4, contours="all").integers()
    rb = suite.evaluate(t, p, 4, contours="all").integers()
    for key in ra:
        assert np.array_equal(ra[key].view(np.uint8), rb[key].view(np.uint8)), key


def test_suite_all_mode(cuda, monkeypatch):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = synth.layered_pair(12, 64, 128, 6, seed=71, noise=0.01)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    res = suite.evaluate(t, p, 6, contours="all")
    assert res.contour_mode == "all" and suite.evaluate(t, p, 6).contour_mode == "first"
    m, mh = res.metrics(), res.metrics_host()
    assert set(m) == set(suite.evaluate(t, p, 6, contours=True).metrics())
    for key in mh:
        np.testing.assert_array_equal(m[key], mh[key], err_msg=key)
    # the device values are the oracle's
    out = _all_pass(t, p, 6)
    ref = _check(yt, yp, 6, out)
    for key in ("hausdorff_distance", "hausdorff_distance_95", "assd"):
        np.testing.assert_array_equal(m[key], ref[key], err_msg=key)
    host = suite.evaluate_host(yt, yp, 6, contours="all", chunk_items=5)
    assert host.contour_mode == "all"
    mhost = host.metrics()
    for key in m:
        np.testing.assert_array_equal(mhost[key], m[key], err_msg=key)
    np.testing.assert_array_equal(host.totals_host(), res.totals_host())
    # chunked contour stage: same results
    monkeypatch.setattr(suite, "CONTOUR_CHUNK_BYTES", 6 * 2 * suite.default_max_pts_all(128) * 4 * 2 * 5)
    chunked = suite.evaluate(t, p, 6, contours="all")
    for key, v in chunked.integers().items():
        assert np.array_equal(v, res.integers()[key]), key
    torch.cuda.synchronize()


def test_kernel_launches(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, _lib
    yt, yp = synth.lesion_pair(4, 96, 128, 4, seed=81, single_blob_interior=False)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    with _lib.kernel_profile() as prof:
        suite.evaluate(t, p, 4, contours=True).metrics()
        torch.cuda.synchronize()
    assert "contour_all_vertices_kernel" not in prof.kernels
    with _lib.kernel_profile() as prof:
        suite.evaluate(t, p, 4, contours="all").metrics()
        torch.cuda.synchronize()
    assert prof.kernels["contour_all_vertices_kernel"][0] == 1
    with pytest.raises(ValueError, match="contours"):
        suite.evaluate(t, p, 4, contours="every")
