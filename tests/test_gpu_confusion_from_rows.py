"""GPU parity: confusion matrices of the certified label pass, bit for bit against numpy, on both count sources.

Seed policy 1 (a mostly accepted stream): the strip kernel runs without its per-pixel histogram; the counts of items whose
two maps are in class order come from the boundary rows (confusion_from_rows_kernel), those of the other items from a
per-pixel histogram (confusion_fix_kernel).  Seed policy 2 (a mostly rejected stream): the strip kernel's histogram."""
import numpy as np
import pytest

from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

pytestmark = pytest.mark.gpu

POLICIES = (1, 2)


@pytest.fixture
def policy(request):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    lib = _lib.load()
    before = lib.octm_label_pass_seed_policy(request.param)
    yield request.param
    lib.octm_label_pass_seed_policy(before)


def _numpy_counts(yt, yp, k):
    """[n, k, k] counts; pixels with a label >= k in either map are not counted.  On the strip kernel's shapes
    (W % 16 == 0, K <= 8) a 128-column strip of an item that holds a label >= 8 is not counted at all."""
    out = np.zeros((yt.shape[0], k, k), np.uint64)
    strips = yt.shape[2] % 16 == 0 and k <= 8
    for i in range(yt.shape[0]):
        keep = (yt[i] < k) & (yp[i] < k)
        if strips:
            for x0 in range(0, yt.shape[2], 128):
                if (yt[i][:, x0:x0 + 128] >= 8).any() or (yp[i][:, x0:x0 + 128] >= 8).any():
                    keep[:, x0:x0 + 128] = False
        t, p = yt[i].astype(np.int64)[keep], yp[i].astype(np.int64)[keep]
        out[i] = np.bincount(t * k + p, minlength=k * k).reshape(k, k)
    return out


def _unsorted(yt, yp):
    dt = (np.diff(yt.astype(np.int16), axis=1) < 0).any(axis=(1, 2))
    dp = (np.diff(yp.astype(np.int16), axis=1) < 0).any(axis=(1, 2))
    return dt.astype(np.uint32) | (dp.astype(np.uint32) << 1)


def _check(yt, yp, k, cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    t, p = torch.as_tensor(yt).to(cuda), torch.as_tensor(yp).to(cuda)
    with _lib.kernel_profile() as prof:
        out = suite.label_pass(t, p, k, counts=True, columns=True, seeds=True, boundaries=True, certify=True)
        torch.cuda.synchronize()
    got = out.counts.cpu().numpy().view(np.uint64)
    want = _numpy_counts(yt, yp, k)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got.sum(axis=0), want.sum(axis=0))         # dataset totals
    uns = out.unsorted.cpu().numpy().view(np.uint32)
    assert (uns & ~np.uint32(3)).sum() == 0                                      # only bits 0 and 1 reach the caller
    if yt.shape[1] <= 500:                        # (the certificate compares labels below 8 only)
        small = ((yt < 8) & (yp < 8)).all(axis=(1, 2))
        np.testing.assert_array_equal(uns[small], _unsorted(yt, yp)[small])
    return set(prof.kernels), uns


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
def test_clean_layered_and_absent_classes(cuda, policy):
    yt, yp = synth.layered_pair(6, 496, 512, 8, seed=31)
    yt[0][yt[0] == 5] = 6                 # class 5 absent from an item (columns stay in class order)
    yp[1][yp[1] == 3] = 4
    yp[1][yp[1] == 0] = 1                 # ... and class 0
    sub = yt[2][:, :100]
    sub[sub == 2] = 3                     # class 2 absent from some columns only
    yp[3][:, 200:][yp[3][:, 200:] == 7] = 6
    kernels, uns = _check(yt, yp, 8, cuda)
    assert (uns == 0).all()
    if policy == 1:
        assert "confusion_from_rows_kernel" in kernels and "confusion_fix_kernel" in kernels
    else:
        assert "confusion_from_rows_kernel" not in kernels and "confusion_fix_kernel" not in kernels


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
@pytest.mark.parametrize("shape", [(4, 62, 128, 5), (3, 37, 64, 3), (3, 128, 144, 4), (2, 96, 2048, 7), (3, 1, 16, 2)])
def test_clean_layered_other_k(cuda, policy, shape):
    n, h, w, k = shape
    yt, yp = synth.layered_pair(n, h, w, k, seed=h + w + k, min_gap=1)
    _check(yt, yp, k, cuda)


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
@pytest.mark.parametrize("noise", [2e-5, 2e-3])
def test_stray_pixels(cuda, policy, noise):
    yt, yp = synth.layered_pair(8, 496, 512, 8, seed=int(noise * 1e6), noise=noise)
    _check(yt, yp, 8, cuda)


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
def test_ragged_and_uniform_random(cuda, policy):
    yt, yp = synth.ragged_pair_device(4, 496, 512, 8, seed=41, device=cuda)
    _check(yt.cpu().numpy(), yp.cpu().numpy(), 8, cuda)
    yt, yp = synth.random_pair(4, 496, 512, 8, seed=42)
    _check(yt, yp, 8, cuda)
    yt, yp = synth.random_pair(3, 62, 128, 5, seed=43)
    _check(yt, yp, 5, cuda)


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
@pytest.mark.parametrize("k,bad", [(8, 9), (8, 255), (6, 7), (5, 5), (3, 200)])
def test_label_at_or_above_k(cuda, policy, k, bad):
    """A label >= K anywhere -- also at the bottom of a column, where the column stays in class order -- leaves the
    item's counts short of H * W, and evaluate(validate=True) raises."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    h, w = 62, 384
    yt, yp = synth.layered_pair(4, h, w, k, seed=51 + k, min_gap=1)
    yp[1, h - 1, 137] = bad               # bottom row: the column is still non-decreasing
    yt[2, h - 1, 100:300] = bad           # part of the bottom row of y_true, across two strips
    yp[3, 10, 5] = bad                    # inside a column: also out of order when bad < the labels below
    _check(yt, yp, k, cuda)
    got = suite.label_pass(torch.as_tensor(yt).to(cuda), torch.as_tensor(yp).to(cuda), k, seeds=True, boundaries=True,
                           certify=True).counts.cpu().numpy()
    assert got[0].sum() == h * w and all(got[i].sum() < h * w for i in (1, 2, 3))
    a, b = torch.as_tensor(yt).to(cuda), torch.as_tensor(yp).to(cuda)
    with pytest.raises(ValueError):
        suite.evaluate(a, b, k, validate=True).totals_host()
    ok = suite.evaluate(a[:1], b[:1], k, validate=True)
    ok.totals_host()


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
def test_tall_and_unaligned_widths(cuda, policy):
    yt, yp = synth.layered_pair(2, 520, 256, 8, seed=61)          # taller than 500 rows: always reported unsorted
    kernels, uns = _check(yt, yp, 8, cuda)
    assert (uns == 3).all()
    yt, yp = synth.layered_pair(3, 100, 200, 8, seed=62, min_gap=1)   # W % 16 != 0: not the strip kernel
    _check(yt, yp, 8, cuda)
    yt, yp = synth.layered_pair(3, 64, 100, 6, seed=63, min_gap=1, noise=0.01)
    _check(yt, yp, 6, cuda)


@pytest.mark.parametrize("policy", POLICIES, indirect=True)
def test_mixed_batch(cuda, policy):
    """Certified, rejected and bad-label items side by side: each gets its counts from the right kernel."""
    a = synth.layered_pair(5, 496, 512, 8, seed=71)
    b = synth.layered_pair(4, 496, 512, 8, seed=72, noise=2e-3)
    c = synth.random_pair(2, 496, 512, 8, seed=73)
    yt = np.concatenate([a[0], b[0], c[0]])
    yp = np.concatenate([a[1], b[1], c[1]])
    order = np.random.default_rng(74).permutation(len(yt))
    yt, yp = yt[order].copy(), yp[order].copy()
    yt[3, 495, 100:110] = 8
    yp[order.tolist().index(0), 495, 511] = 255     # a clean item with one bad label (its columns stay in order)
    _, uns = _check(yt, yp, 8, cuda)
    assert (uns == 0).sum() >= 3 and (uns != 0).sum() >= 6


def test_policies_agree_through_the_suite(cuda):
    """evaluate() integers are the same with either count source (and with the data-following default)."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    lib = _lib.load()
    yt, yp = synth.layered_pair(6, 496, 512, 8, seed=81)
    yp[4] = synth.layered_pair(1, 496, 512, 8, seed=82, noise=2e-3)[1][0]
    a, b = torch.as_tensor(yt).to(cuda), torch.as_tensor(yp).to(cuda)
    before = lib.octm_label_pass_seed_policy(-1)
    runs = []
    try:
        for pol in (1, 2, 0):
            lib.octm_label_pass_seed_policy(pol)
            runs.append(suite.evaluate(a, b, 8).integers())
    finally:
        lib.octm_label_pass_seed_policy(before)
    np.testing.assert_array_equal(runs[0]["confusion"], _numpy_counts(yt, yp, 8))
    for r in runs[1:]:
        assert r.keys() == runs[0].keys()
        for name in r:
            np.testing.assert_array_equal(r[name], runs[0][name], err_msg=name)
