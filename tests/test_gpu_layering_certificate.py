"""GPU parity: the label pass's layering certificate (``unsorted[i]`` bit m = some column of map m is not
non-decreasing from top to bottom) against numpy, on both kernels; it decides whether a contour may be measured from the
boundary rows alone, so a false "sorted" would be a silent wrong result."""
import numpy as np
import pytest

from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

pytestmark = pytest.mark.gpu


def _expected(yt, yp, tall_limit=500, fast=True):
    out = np.zeros(len(yt), np.uint32)
    for i in range(len(yt)):
        for m, a in enumerate((yt[i], yp[i])):
            if (np.diff(a.astype(np.int16), axis=0) < 0).any():
                out[i] |= 1 << m
    if fast and yt.shape[1] > tall_limit:
        out[:] = 3                                  # the strip kernel does not certify items taller than 500 rows
    return out


def _run(yt, yp, k, cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    t, p = torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda)
    lp = suite.label_pass(t, p, k, seeds=True, boundaries=True, certify=True)
    fast = bool(_lib.load().octm_label_pass_path(yt.shape[1], yt.shape[2], k, t.data_ptr(), p.data_ptr()))
    return lp.unsorted.cpu().numpy().view(np.uint32), fast


@pytest.mark.parametrize("shape,k", [((6, 496, 512), 8), ((5, 124, 256), 6), ((4, 62, 128), 3), ((3, 496, 1024), 8),
                                     ((4, 63, 96), 8), ((5, 33, 50), 8), ((3, 64, 128), 12), ((2, 600, 256), 5)])
def test_certificate_matches_numpy(cuda, shape, k):
    n, h, w = shape
    rng = np.random.default_rng(h * w + k)
    yt, yp = synth.layered_pair(n, h, w, k, seed=11 + k)
    # item 0: clean.  others: single defects of every kind the two-part check has to catch
    if n > 1:
        yp[1, h // 2, w // 3] = (yp[1, h // 2, w // 3] + 1) % k                     # one stray pixel
    if n > 2:
        x = w - 5
        col = yt[2, :, x].copy()
        r = int(np.argmax(col > 0))                                                  # first row of class >= 1
        if 1 <= r < h - 2:
            yt[2, r, x], yt[2, r + 1, x] = col[r - 1], col[r]                         # ... 0 1 -> 0 0? keep order: no-op-safe
            yt[2, r - 1, x] = col[r]                                                 # swap across the boundary: 1 above 0
    if n > 3:
        yt[3, 0, 0] = k - 1                                                          # largest label in the very first row
    if n > 4:
        yp[4, h - 1, w - 1] = 0                                                      # smallest label in the very last row
    if n > 5:
        rows = rng.integers(1, h - 1, size=8)
        yt[5, rows, rng.integers(0, w, size=8)] = rng.integers(0, k, size=8)         # sparse salt in y_true only
    got, fast = _run(yt, yp, k, cuda)
    np.testing.assert_array_equal(got, _expected(yt, yp, fast=fast))
    assert got[0] == (3 if (fast and h > 500) else 0)


def test_interleaving_defects(cuda):
    """Defects that keep BOTH row parities in order and are only visible in how they interleave (part 2 of the
    check): rows 2r and 2r+1 exchanged around a boundary."""
    k, h, w = 8, 496, 512
    yt, yp = synth.layered_pair(4, h, w, k, seed=77)
    for i, x in ((1, 7), (2, 200), (3, 511)):
        col = yt[i, :, x]
        r = int(np.argmax(col >= 3))                      # first row of class >= 3: rows r-1 | r differ
        a, b = col[r - 1], col[r]
        yt[i, r - 1, x], yt[i, r, x] = b, a               # adjacent exchange: each parity chain stays monotone
    got, _ = _run(yt, yp, k, cuda)
    np.testing.assert_array_equal(got, _expected(yt, yp))
    assert got[0] == 0 and all(got[1:] & 1)


def test_random_maps_are_never_certified(cuda):
    yt, yp = synth.random_pair(3, 124, 256, 8, seed=5)
    got, _ = _run(yt, yp, 8, cuda)
    assert (got == 3).all()
    z = np.zeros((2, 64, 128), np.uint8)                  # constant maps are sorted
    got, _ = _run(z, z, 4, cuda)
    assert (got == 0).all()


def test_verified_pairs_do_not_depend_on_max_pts_and_wide_images_need_no_retry(cuda):
    """A pair with two certified sides is measured from the boundary rows and stores nothing: max_pts (what is STORED per
    contour) must not matter.  Noisy pairs with a tiny bound go through the overflow retry and end with the same numbers.
    A 1024-wide B-scan (2 W + sum |dh| > 2048 vertices per contour) must not overflow with the default bound."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, synth
    for noise in (0.0, 1e-4):
        yt, yp = synth.layered_pair(5, 496, 512, 8, seed=31, noise=noise)
        t, p = torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda)
        a = suite.evaluate(t, p, 8, max_pts=2048)
        b = suite.evaluate(t, p, 8, max_pts=256)
        ma, mb = a.metrics(), b.metrics()
        # integers bit-exact; the float64 distance sums are added in a path-dependent order (1e-12 relative)
        for name in ("hausdorff_distance", "hausdorff_distance_95"):
            np.testing.assert_array_equal(ma[name], mb[name], err_msg=f"{name} noise {noise}")
        np.testing.assert_allclose(ma["assd"], mb["assd"], rtol=1e-12, atol=0, err_msg=f"assd noise {noise}")
        ia, ib = a.integers(), b.integers()
        for name in ("contour_max_sq", "contour_p95_sq"):
            np.testing.assert_array_equal(ia[name], ib[name], err_msg=f"{name} noise {noise}")
        np.testing.assert_allclose(ia["contour_sum_dist"], ib["contour_sum_dist"], rtol=1e-12, atol=0)
        if noise == 0.0:
            assert int(ib["contour_n_pts"].max()) > 256                          # longer than the bound, and still exact
    yt, yp = synth.layered_pair(3, 496, 1024, 10, seed=32, noise=0.0)
    t, p = torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda)
    with_default = suite.evaluate(t, p, 10)
    assert with_default.contours.max_pts == 4096
    ref = suite.evaluate(t, p, 10, max_pts=8192)
    for name in ("hausdorff_distance", "hausdorff_distance_95", "assd"):
        np.testing.assert_allclose(with_default.metrics()[name], ref.metrics()[name], rtol=1e-12, atol=0, err_msg=name)
    assert int(with_default.integers()["contour_n_pts"].max()) > 2048
