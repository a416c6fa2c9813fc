"""GPU parity: fused label pass (K1 + K2 + K3 + seeds) against the oracle -- bit-exact integers."""
import numpy as np
import pytest

from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

pytestmark = pytest.mark.gpu


def _first_pos_oracle(lab, k):
    flat = lab.reshape(lab.shape[0], -1)
    out = np.full((lab.shape[0], k), 0xFFFFFFFF, np.uint32)
    for i in range(lab.shape[0]):
        for c in range(k):
            idx = np.flatnonzero(flat[i] == c)
            if idx.size:
                out[i, c] = idx[0]
    return out


def _run(yt, yp, k, cuda, boundaries=True, certify=False):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    t, p = torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda)
    out = suite.label_pass(t, p, k, counts=True, columns=True, seeds=True, boundaries=boundaries, certify=certify)
    torch.cuda.synchronize()
    return out


def _check(yt, yp, k, cuda):
    # certify=False: seeds tracked pixel by pixel; certify=True (the suite's call): seeds from the column totals on maps
    # in class order, from a rescan on the others -- same outputs either way
    _check_one(yt, yp, k, cuda, False)
    _check_one(yt, yp, k, cuda, True)


def _check_one(yt, yp, k, cuda, certify):
    out = _run(yt, yp, k, cuda, certify=certify)
    n = yt.shape[0]
    ref = [lo.score_bscan_fast(yt[i], yp[i], k) for i in range(n)]
    np.testing.assert_array_equal(out.counts.cpu().numpy().view(np.uint64), np.stack([r["confusion"] for r in ref]))
    np.testing.assert_array_equal(out.thick_absdiff.cpu().numpy(), np.stack([r["thickness_absdiff"] for r in ref]))
    np.testing.assert_array_equal(out.bnd_sq.cpu().numpy(), np.stack([r["boundary_sq"] for r in ref]))
    np.testing.assert_array_equal(out.bnd_abs.cpu().numpy(), np.stack([r["boundary_abs"] for r in ref]))
    np.testing.assert_array_equal(out.bnd_true.cpu().numpy(), np.stack([r["boundary_true"] for r in ref]))
    np.testing.assert_array_equal(out.bnd_pred.cpu().numpy(), np.stack([r["boundary_pred"] for r in ref]))
    fp = out.first_pos.cpu().numpy().view(np.uint32)
    np.testing.assert_array_equal(fp[:, 0], _first_pos_oracle(yt, k))
    np.testing.assert_array_equal(fp[:, 1], _first_pos_oracle(yp, k))
    if certify and yt.shape[1] <= 500:          # (the strip kernel reports taller items unsorted without looking)
        want = ((np.diff(yt.astype(np.int16), axis=1) < 0).any(axis=(1, 2)).astype(np.uint32)
                | ((np.diff(yp.astype(np.int16), axis=1) < 0).any(axis=(1, 2)).astype(np.uint32) << 1))
        np.testing.assert_array_equal(out.unsorted.cpu().numpy().view(np.uint32), want)


def test_golden_suite(cuda, golden_dir):
    g = np.load(f"{golden_dir}/suite_golden.npz")
    for name in g["names"]:
        yt, yp, k = g[f"{name}/y_true"], g[f"{name}/y_pred"], int(g[f"{name}/K"])
        out = _run(yt, yp, k, cuda)
        np.testing.assert_array_equal(out.counts.cpu().numpy().view(np.uint64), g[f"{name}/confusion"], err_msg=name)
        np.testing.assert_array_equal(out.thick_absdiff.cpu().numpy(), g[f"{name}/thickness_absdiff"], err_msg=name)
        np.testing.assert_array_equal(out.bnd_sq.cpu().numpy(), g[f"{name}/boundary_sq"], err_msg=name)
        np.testing.assert_array_equal(out.bnd_abs.cpu().numpy(), g[f"{name}/boundary_abs"], err_msg=name)
        np.testing.assert_array_equal(out.bnd_true.cpu().numpy(), g[f"{name}/boundary_true"], err_msg=name)
        np.testing.assert_array_equal(out.bnd_pred.cpu().numpy(), g[f"{name}/boundary_pred"], err_msg=name)


@pytest.mark.parametrize("shape", [(3, 496, 512, 8), (2, 496, 768, 8), (2, 62, 128, 5), (5, 37, 64, 3),
                                   (1, 1, 16, 2), (2, 3, 2048, 7), (1, 1030, 256, 8), (3, 128, 144, 4)])
def test_fast_kernel_layered_and_random(cuda, shape):
    """Shapes the TMA-staged kernel takes (W % 16 == 0, K <= 8): layered + salt noise, and uniform random."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    n, h, w, k = shape
    assert _lib.load().octm_label_pass_path(h, w, k, 0, 0) == 1
    if h >= 16:
        yt, yp = synth.layered_pair(n, h, w, k, seed=h * w + k, noise=0.03, min_gap=1)
        _check(yt, yp, k, cuda)
    yt, yp = synth.random_pair(n, h, w, k, seed=7 * h + w)
    _check(yt, yp, k, cuda)


@pytest.mark.parametrize("shape", [(2, 33, 50, 16), (3, 17, 23, 2), (1, 496, 1024, 10), (2, 21, 300, 12), (2, 5, 7, 9), (1, 1, 1, 2),
                                   (2, 64, 96, 11), (2, 33, 52, 16), (3, 70, 132, 9), (1, 600, 260, 13), (40, 9, 4, 10),
                                   (2, 1, 128, 16), (2, 496, 500, 8)])
def test_generic_kernel(cuda, shape):
    """Ragged widths and K > 8 go through the generic kernel."""
    n, h, w, k = shape
    yt, yp = synth.random_pair(n, h, w, k, seed=h + 31 * w)
    _check(yt, yp, k, cuda)
    if h >= 32:
        yt, yp = synth.layered_pair(n, h, w, k, seed=h * w, noise=0.02, min_gap=1)
        _check(yt, yp, k, cuda)


def test_many_items_persistent_grid(cuda):
    """More items than resident CTAs: the persistent loop and the ring must stay in step across items."""
    yt, yp = synth.layered_pair(700, 40, 64, 6, seed=99, noise=0.05, min_gap=1)
    _check(yt, yp, 6, cuda)


def test_uniform_and_absent_classes(cuda):
    """All-one-class maps and classes that never occur (first_pos = NO_SEED, zero rows in cm)."""
    yt = np.zeros((2, 24, 32), np.uint8)
    yp = np.full((2, 24, 32), 3, np.uint8)
    yt[1, 5:9, 3:20] = 2
    _check(yt, yp, 5, cuda)


def test_standalone_confusion_any_shape(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    rng = np.random.default_rng(3)
    for shape, k in [((4, 253952), 8), ((3, 1000), 16), ((2, 7, 9, 11), 4), ((5, 4096), 2)]:
        a = rng.integers(0, k, size=shape, dtype=np.uint8)
        b = rng.integers(0, k, size=shape, dtype=np.uint8)
        cm = suite.confusion(torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda), k).cpu().numpy()
        for i in range(shape[0]):
            np.testing.assert_array_equal(cm[i].astype(np.uint64), lo.confusion_matrix(a[i], b[i], k))


def test_boundary_error_kernel(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    rng = np.random.default_rng(4)
    bt = rng.integers(0, 496, size=(6, 9, 1024), dtype=np.int32)
    bp = bt + rng.integers(-7, 8, size=bt.shape, dtype=np.int32)
    sq, ab = suite.boundary_error(torch.from_numpy(bt).to(cuda), torch.from_numpy(bp).to(cuda))
    d = bt.astype(np.int64) - bp
    np.testing.assert_array_equal(sq.cpu().numpy(), (d * d).sum(-1))
    np.testing.assert_array_equal(ab.cpu().numpy(), np.abs(d).sum(-1))


def test_derived_ratios_match_oracle(cuda):
    """float64 ratios from GPU counts vs the per-class reference-style oracle: 1e-6 relative (0 ulp expected)."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = synth.layered_pair(2, 96, 128, 6, seed=5, noise=0.02)
    res = suite.evaluate(torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda), 6, contours=False)
    m = res.metrics()
    for i in range(2):
        ref = lo.score_bscan(yt[i], yp[i], 6, contours=False)
        for name in lo.COUNT_METRICS + ("thickness_difference", "boundary_mse", "boundary_rmse", "boundary_mad"):
            np.testing.assert_allclose(m[name][i], ref[name], rtol=1e-6, atol=0, err_msg=name)
            assert np.array_equal(m[name][i], ref[name]), name      # in practice bit-identical


@pytest.mark.parametrize("shape", [(600, 9, 4, 10), (300, 33, 132, 16), (150, 70, 520, 9), (1200, 1, 128, 16), (80, 120, 1024, 10),
                                   (700, 17, 52, 12), (640, 40, 100, 8)])
def test_wide_kernel(cuda, shape):
    """K <= 16, W % 4 == 0 and enough strips of work (>= 4 per SM): label_pass_wide (run queues drained in lockstep)"""
    n, h, w, k = shape
    assert n * ((w + 127) // 128) >= 592
    yt, yp = synth.random_pair(n, h, w, k, seed=h + 31 * w)
    _check(yt, yp, k, cuda)
    if h >= 2 * k:
        yt, yp = synth.layered_pair(n, h, w, k, seed=h * w, noise=0.02, min_gap=1)
        _check(yt, yp, k, cuda)
        yt, yp = synth.layered_pair(n, h, w, k, seed=h * w + 1, noise=0.0, min_gap=1)     # clean: certificate says sorted
        _check(yt, yp, k, cuda)


def test_wide_and_bytewise_kernels_agree_on_paths_and_results(cuda):
    """K > 8: W % 4 == 0 takes the warp-per-strip kernel (path 2), other widths and unaligned views the byte-wise one (0)"""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    lib = _lib.load()
    assert lib.octm_label_pass_path(496, 1024, 10, 0, 0) == 2
    assert lib.octm_label_pass_path(496, 1022, 10, 0, 0) == 0
    assert lib.octm_label_pass_path(496, 512, 8, 0, 0) == 1
    yt, yp = synth.layered_pair(250, 120, 264, 10, seed=77, noise=0.02, min_gap=1)     # 750 strips: the wide kernel
    yt[1, 5, 7] = 200                                       # a label >= K: dropped, never aliased
    yp[2, 100, 263] = 16
    yp[3, 0, 0] = 11
    a = suite.label_pass(torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda), 10, counts=True, columns=True, seeds=True,
                         boundaries=True, certify=True)
    # the same maps as unaligned views (offset by one byte): the byte-wise kernel
    buf_t = torch.zeros(yt.size + 1, dtype=torch.uint8, device=cuda)
    buf_p = torch.zeros(yp.size + 1, dtype=torch.uint8, device=cuda)
    buf_t[1:] = torch.from_numpy(yt).to(cuda).reshape(-1)
    buf_p[1:] = torch.from_numpy(yp).to(cuda).reshape(-1)
    vt, vp = buf_t[1:].view(yt.shape), buf_p[1:].view(yp.shape)
    assert lib.octm_label_pass_path(120, 264, 10, vt.data_ptr(), vp.data_ptr()) == 0
    b = suite.label_pass(vt, vp, 10, counts=True, columns=True, seeds=True, boundaries=True, certify=True)
    for name in ("counts", "thick_absdiff", "bnd_sq", "bnd_abs", "bnd_true", "bnd_pred", "first_pos", "unsorted"):
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x, y), name
    assert int(a.counts[1].sum()) == 120 * 264 - 1


def test_seed_policies_give_the_same_seeds(cuda):
    """The strip kernel's seeds come from the column totals (+ a rescan of rejected maps) or from per-pixel tracking,
    chosen by the data; both must match the oracle and each other, on clean, noisy and random maps."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    lib = _lib.load()
    before = lib.octm_label_pass_seed_policy(-1)
    try:
        for policy in (1, 2, 0):
            lib.octm_label_pass_seed_policy(policy)
            assert lib.octm_label_pass_seed_policy(-1) == policy
            for noise in (0.0, 0.02):
                yt, yp = synth.layered_pair(5, 496, 512, 8, seed=11 + policy, noise=noise, min_gap=1)
                _check_one(yt, yp, 8, cuda, True)
            yt, yp = synth.random_pair(3, 62, 128, 5, seed=12)
            _check_one(yt, yp, 5, cuda, True)
        # following the data: a rejected batch switches the next call to per-pixel tracking (no rescan kernel), a clean
        # batch switches back; the outputs never depend on it
        lib.octm_label_pass_seed_policy(0)
        yt, yp = synth.layered_pair(6, 496, 512, 8, seed=21, noise=0.01, min_gap=1)
        t, p = torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda)
        ct, cp = torch.from_numpy(synth.layered_pair(6, 496, 512, 8, seed=22)[0]).to(cuda), None
        cp = ct.clone()

        def kernels(a, b):
            with _lib.kernel_profile() as prof:
                out = suite.label_pass(a, b, 8, counts=True, columns=True, seeds=True, boundaries=True, certify=True)
                torch.cuda.synchronize()
            return out, set(prof.kernels)

        kernels(ct, cp)                                     # clean report
        o1, k1 = kernels(t, p)                              # decided by the clean report: totals + rescan
        assert "first_pos_fix_kernel" in k1
        o2, k2 = kernels(t, p)                              # decided by the noisy report: per pixel
        assert "first_pos_fix_kernel" not in k2
        assert torch.equal(o1.first_pos, o2.first_pos) and torch.equal(o1.unsorted, o2.unsorted)
        assert torch.equal(o1.counts, o2.counts) and torch.equal(o1.bnd_pred, o2.bnd_pred)
        _, k3 = kernels(ct, cp)                             # still per pixel (the report before was noisy) ...
        _, k4 = kernels(ct, cp)                             # ... and back
        assert "first_pos_fix_kernel" not in k3 and "first_pos_fix_kernel" in k4
    finally:
        lib.octm_label_pass_seed_policy(before)
