"""GPU parity of the whole suite (``suite.evaluate``, contour ``[0]``) with the oracle at the geometries where the
kernels branch on shape, class count or batch size: tall B-scans (Cirrus and Topcon heights), odd, unaligned and very
wide widths, 11 to 16 classes, squared distances beyond the shared-memory counters, contours at the 16-bit counter
width, the 4095 / 4096 / 8192-row envelope, batches of hundreds of items and the chunked contour stage.

The kernels route on device data, so no route is observable from outside; every case asserts instead the input
property that forces its route (row count, label-pass path code, oracle maximum D2, vertex count), so that a change of
the inputs cannot silently move a case off its branch.  Cases A to D run under seed policy 1, policy 2, and policy 0
twice in a row (the second call follows the report the first one left)."""
import numpy as np
import pytest
import torch

from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite, synth

import geometry_oracle as go

pytestmark = pytest.mark.gpu

POLICIES = (1, 2, 0, 0)
SHORT_ROWS = 500                 # the strip label kernel certifies items of at most this many rows
WIDE_COUNT_LIMIT = 1024 << 11    # PASS 2 counts squared distances below this in shared memory
FUSED = "layered_distance_kernel"


@pytest.fixture(scope="module")
def lib(cuda):
    lib = _lib.load()
    before = lib.octm_label_pass_seed_policy(-1)
    yield lib
    lib.octm_label_pass_seed_policy(before)


def _dev(a, cuda):
    return a.to(cuda) if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else a


def _evaluate(t, p, k, **kw):
    """evaluate() with every liboctm launch recorded; the results are read inside the profile (overflow retry)."""
    with _lib.kernel_profile() as prof:
        res = suite.evaluate(t, p, k, boundaries=True, **kw)
        res.integers()
        torch.cuda.synchronize()
    return res, prof.kernels


def _fused_ran(kernels):
    return any(name.startswith(FUSED) for name in kernels)


def _path(lib, t, p, k):
    return int(lib.octm_label_pass_path(t.shape[1], t.shape[2], k, t.data_ptr(), p.data_ptr()))


def _expected_unsorted(yt, yp, strip_path):
    """The certificate as the kernels define it: bit m = a column of map m is out of class order; the strip kernel
    certifies no item taller than SHORT_ROWS."""
    out = np.zeros(len(yt), np.uint32)
    for i in range(len(yt)):
        for m, a in enumerate((yt[i], yp[i])):
            if (np.diff(a.astype(np.int16), axis=0) < 0).any():
                out[i] |= 1 << m
    if strip_path and yt.shape[1] > SHORT_ROWS:
        out[:] = 3
    return out


def _under_policies(lib, cuda, yt, yp, k, **kw):
    """The oracle check under every policy of POLICIES; returns [(policy, kernels, result)]."""
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    yt, yp = _host(yt), _host(yp)
    runs = []
    for policy in POLICIES:
        lib.octm_label_pass_seed_policy(policy)
        res, kernels = _evaluate(t, p, k, **kw)
        go.check_suite(yt, yp, k, res)
        runs.append((policy, kernels, res))
    unsorted = runs[0][2].integers()["unsorted"]
    for _, _, res in runs[1:]:
        np.testing.assert_array_equal(res.integers()["unsorted"], unsorted)
    return runs


# ------------------------------------------------------------------------------------------------- A. tall B-scans
def _layered_variants(n, h, w, k, seed, cuda):
    yield "clean", synth.layered_pair(n, h, w, k, seed=seed)
    yield "noise 2e-5", synth.layered_pair(n, h, w, k, seed=seed + 1, noise=2e-5)
    yield "noise 2e-3", synth.layered_pair(n, h, w, k, seed=seed + 2, noise=2e-3)
    yt, yp = synth.ragged_pair_device(n, h, w, k, seed=seed + 3, device=cuda)
    yield "ragged", (yt.cpu().numpy(), yp.cpu().numpy())


@pytest.mark.parametrize("h,w,k", [(1024, 512, 8), (885, 512, 8), (650, 512, 4), (640, 400, 6)])
def test_tall_layered_bscans(cuda, lib, h, w, k):
    """Items taller than 500 rows are never certified: every call after the first sees a stream of rejected maps."""
    for name, (yt, yp) in _layered_variants(2, h, w, k, 100 + h + k, cuda):
        t, p = _dev(yt, cuda), _dev(yp, cuda)
        assert h > SHORT_ROWS and _path(lib, t, p, k) == 1, name
        runs = _under_policies(lib, cuda, yt, yp, k)
        np.testing.assert_array_equal(runs[0][2].integers()["unsorted"], _expected_unsorted(yt, yp, True), err_msg=name)
        assert runs[1][0] == 2 and FUSED + "_rows" in runs[1][1], (name, sorted(runs[1][1]))
        assert runs[0][0] == 1 and FUSED in runs[0][1], (name, sorted(runs[0][1]))
        if name == "clean":         # nothing is walked after the pinned rows-first call: policy 0 keeps that order
            for _, kernels, _ in runs[2:]:
                assert FUSED + "_rows" in kernels, (name, sorted(kernels))


def test_tall_lesion_slices(cuda, lib):
    for single in (True, False):
        yt, yp = synth.lesion_pair(2, 1024, 512, 4, seed=3100 + single, single_blob_interior=single)
        runs = _under_policies(lib, cuda, yt, yp, 4)
        np.testing.assert_array_equal(runs[0][2].integers()["unsorted"], [3, 3])


@pytest.mark.parametrize("h", [500, 501, 504, 505])
def test_heights_around_the_byte_counter_period(cuda, lib, h):
    """The strip kernel flushes its byte counters after 126 four-row groups (rows 501 to 504 end the 126th): 500 rows is
    the last height whose column totals may share the histogram's shared memory and that is certified.  Item 0 clean,
    item 1 noisy."""
    yt, yp = synth.layered_pair(2, h, 512, 8, seed=h)
    _, yp1 = synth.layered_pair(2, h, 512, 8, seed=h, noise=2e-3)
    yp[1] = yp1[1]
    assert _path(lib, _dev(yt, cuda), _dev(yp, cuda), 8) == 1
    runs = _under_policies(lib, cuda, yt, yp, 8)
    got = runs[0][2].integers()["unsorted"]
    np.testing.assert_array_equal(got, _expected_unsorted(yt, yp, True))
    assert got.tolist() == ([0, 2] if h <= SHORT_ROWS else [3, 3])


# ------------------------------------------------------------------------------------------------------- B. widths
# (H, W, K, label-pass path code, fused contour kernel): 1 strip kernel (W % 16 == 0, W <= 2048, K <= 8), 2 the
# 4-byte kernels, 0 the byte-wise one; the fused kernel needs an even width
WIDTHS = [(496, 500, 8, 2, True), (496, 511, 8, 0, False), (496, 2048, 8, 1, True), (64, 2056, 6, 2, True),
          (2, 512, 3, 1, True), (512, 2, 3, 0, True)]


@pytest.mark.parametrize("h,w,k,path,fused", WIDTHS)
def test_widths(cuda, lib, h, w, k, path, fused):
    yt, yp = synth.layered_pair(3, h, w, k, seed=h + w, noise=2e-3)
    yt[2], yp[2] = synth.layered_pair(1, h, w, k, seed=h + w + 1)
    if min(h, w) == 2:                                      # random labels give a map full of small contours
        rt, rp = synth.random_pair(2, h, w, k, seed=h * w)
        yt = np.concatenate([yt, rt])
        yp = np.concatenate([yp, rp])
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    assert _path(lib, t, p, k) == path
    runs = _under_policies(lib, cuda, yt, yp, k)
    for policy, kernels, res in runs:
        assert _fused_ran(kernels) == fused, (policy, sorted(kernels))
    np.testing.assert_array_equal(runs[0][2].integers()["unsorted"], _expected_unsorted(yt, yp, path == 1))


# ------------------------------------------------------------------------------------------------------ C. classes
def _stray_blob_items(h, w, k, seed):
    """Clean layered items where class 1 (the class after pixel (0, 0)'s) fails verification in one map: a stray
    blob of class 1 above its layer, in y_pred (item 0) or y_true (item 1); item 2 has it in a deep column of the
    top layer, below the layer's shallowest row."""
    yt, yp = synth.layered_pair(3, h, w, k, seed=seed)
    yp[0, 4:7, w // 3:w // 3 + 5] = 1
    yt[1, 2, w - 9] = 1
    bnd = lo.boundaries(yt[2], k)[0]
    x = int(np.argmax(bnd))
    assert bnd[x] - 3 > bnd.min()
    yt[2, bnd[x] - 3, x] = 1
    for i in range(3):
        assert yt[i, 0, 0] == 0 and yp[i, 0, 0] == 0
    return yt, yp


@pytest.mark.parametrize("k", [11, 12, 13, 16])
@pytest.mark.parametrize("w", [512, 1024])
def test_many_classes(cuda, lib, k, w):
    for noise in (0.0, 2e-3):
        yt, yp = synth.layered_pair(2, 496, w, k, seed=k * w + int(noise * 1e4), noise=noise)
        _under_policies(lib, cuda, yt, yp, k)
    yt, yp = _stray_blob_items(496, w, k, seed=k + w)
    runs = _under_policies(lib, cuda, yt, yp, k)
    assert all(_fused_ran(kernels) for _, kernels, _ in runs)
    np.testing.assert_array_equal(runs[0][2].integers()["unsorted"], [2, 1, 1])


# ------------------------------------------------------------------------------------------------ D. far distances
def test_prediction_rolled_beyond_the_wide_counters(cuda, lib):
    """Every layer of the prediction 760 rows below the truth: squared distances past PASS 2's counters."""
    h, w, k, shift = 1024, 512, 3, 760
    rng = np.random.default_rng(5)
    x = np.arange(w)
    items = []
    for i in range(2):
        b1 = 90 + np.rint(20 * np.sin(2 * np.pi * x / rng.uniform(300, 900) + rng.uniform(0, 6))).astype(np.int64)
        bt = np.stack([b1, b1 + 40 + i * 10])[None]
        items.append((lo.labels_from_boundaries(bt, h)[0], lo.labels_from_boundaries(bt + shift, h)[0]))
    yt = np.stack([a for a, _ in items])
    yp = np.stack([b for _, b in items])
    for i in range(2):
        assert go.max_sq(yt[i], yp[i], k) >= WIDE_COUNT_LIMIT
    _under_policies(lib, cuda, yt, yp, k)


@pytest.mark.parametrize("h,w", [(496, 512), (512, 512), (1024, 1024)])
def test_single_stray_pixels_far_from_their_layer(cuda, lib, h, w):
    """A stray pixel hands its pair on with vmax = 4 (H^2 + W^2): below the counter limit at 496x512 (wide counting),
    at or above it from 512x512 on (vertex-list search)."""
    k = 6
    yt, yp = synth.layered_pair(3, h, w, k, seed=h + 7 * w)
    yp[0, 3, w - 3] = 4                     # far above layer 4
    yt[1, h - 2, 1] = 1                     # far below layer 1
    yp[2, 2, 2] = k - 1
    yt[2, h - 3, w - 2] = 2
    assert (4 * (h * h + w * w) < WIDE_COUNT_LIMIT) == (h == 496)
    assert _path(lib, _dev(yt, cuda), _dev(yp, cuda), k) == 1
    runs = _under_policies(lib, cuda, yt, yp, k)
    expected = _expected_unsorted(yt, yp, True)
    np.testing.assert_array_equal(runs[0][2].integers()["unsorted"], expected)
    assert expected.tolist() == ([2, 1, 3] if h <= SHORT_ROWS else [3, 3, 3])


# ------------------------------------------------------------------------------------------------ E. counter width
@pytest.mark.parametrize("shift", [0, 1])
def test_contours_at_the_16_bit_counter_width(cuda, shift):
    """65,535 vertices fit one 16-bit counter (shift 0: every distance is 0); 65,536 are handed on and retried up to
    MAX_MAX_PTS; 65,537 exceed MAX_MAX_PTS and must raise, never return a number."""
    from oracle import contours_oracle as co
    for n_vertices in (65535, 65536, 65537):
        yt, yp = go.sawtooth_pair(128, 1024, n_vertices, shift)
        assert len(co.first_contour_lattice(yt[0] == 0)) == n_vertices
        t, p = _dev(yt, cuda), _dev(yp, cuda)
        if n_vertices > suite.MAX_MAX_PTS:
            with pytest.raises(_lib.OctmError, match=f"more than {suite.MAX_MAX_PTS} vertices: pass a larger max_pts"):
                suite.evaluate(t, p, 2, boundaries=True).integers()
            res, _ = _evaluate(t, p, 2, max_pts=n_vertices + 3)          # what the message asks for
            assert go.check_suite(yt, yp, 2, res) == 2
            continue
        res, _ = _evaluate(t, p, 2)
        assert go.check_suite(yt, yp, 2, res) == 2
        assert res.integers()["contour_n_pts"][0].tolist() == [[n_vertices] * 2] * 2


# ----------------------------------------------------------------------------------------------- F. envelope edges
@pytest.mark.parametrize("h,w,k", [(4095, 64, 4), (4096, 64, 4), (4097, 64, 4), (8192, 16, 3), (16, 8192, 3)])
def test_envelope_edges(cuda, lib, h, w, k):
    """The fused contour path stops above 4095 rows, the strip label kernel above 4096 rows and 2048 columns."""
    yt, yp = synth.layered_pair(2, h, w, k, seed=h + w)
    _, yp1 = synth.layered_pair(2, h, w, k, seed=h + w, noise=1e-3)
    yp[1] = yp1[1]
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    path = _path(lib, t, p, k)
    assert path == (1 if h <= 4096 and w <= 2048 else 2)
    res, kernels = _evaluate(t, p, k)
    go.check_suite(yt, yp, k, res)
    assert _fused_ran(kernels) == (h <= 4095), sorted(kernels)
    np.testing.assert_array_equal(res.integers()["unsorted"], _expected_unsorted(yt, yp, path == 1))


@pytest.mark.parametrize("h,w", [(8193, 16), (16, 8193)])
def test_sides_beyond_8192_are_refused(cuda, h, w):
    yt, yp = synth.layered_pair(1, h, w, 3, seed=h)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    lp = suite.label_pass(t, p, 3, seeds=True, boundaries=True, certify=True)       # the label pass takes this size
    assert np.array_equal(lp.counts[0].cpu().numpy().view(np.uint64), lo.confusion_matrix(yt[0], yp[0], 3))
    with pytest.raises(_lib.OctmError, match="8192"):
        suite.evaluate(t, p, 3)
    with pytest.raises(_lib.OctmError, match="8192"):
        suite.contour_pass(t, p, 3)


# ------------------------------------------------------------------------------------------------ G. large batches
def _check_sample(cuda, yt, yp, k, res, n_sample, seed):
    n = yt.shape[0]
    rng = np.random.default_rng(seed)
    idx = sorted({0, n - 1, *rng.choice(np.arange(1, n - 1), size=n_sample - 2, replace=False).tolist()})
    st, sp = yt[idx].cpu().numpy(), yp[idx].cpu().numpy()
    go.check_suite(st, sp, k, res, items=idx)
    whole = res.integers()
    for j, i in enumerate(idx):
        one, _ = _evaluate(yt[i:i + 1], yp[i:i + 1], k)
        alone = one.integers()
        for key, val in alone.items():
            if key == "contour_sum_dist":
                np.testing.assert_allclose(whole[key][i], val[0], rtol=go.SUM_RTOL, err_msg=str(i))
            else:
                assert np.array_equal(whole[key][i], val[0]), (i, key)


def test_large_batches(cuda):
    sms = torch.cuda.get_device_properties(cuda).multi_processor_count
    k, n = 8, 1024
    yt, yp = synth.layered_pair_device(n, 496, 512, k, seed=801, device=cuda, noise=2e-3)
    rt, rp = synth.ragged_pair_device(n // 4, 496, 512, k, seed=802, device=cuda)
    yt[3::4], yp[3::4] = rt, rp
    assert n * k > 4 * sms                          # more (item, class) pairs than CTAs: the grid strides over them
    res, _ = _evaluate(yt, yp, k)
    _check_sample(cuda, yt, yp, k, res, 24, 803)

    k, n = 10, 160
    yt, yp = synth.layered_pair_device(n, 496, 1024, k, seed=804, device=cuda, noise=2e-3)
    assert n * (1024 // 128) >= 2 * sms * 2         # enough strips for label_pass_wide
    res, kernels = _evaluate(yt, yp, k)
    assert "label_pass_wide" in kernels, sorted(kernels)
    _check_sample(cuda, yt, yp, k, res, 24, 805)


# ---------------------------------------------------------------------------------------- H. chunked "first" mode
def test_chunked_first_mode(cuda, monkeypatch):
    """Chunks slice the seeds, the boundary rows and the certificate.  The clean (certified) items come first, so
    that they line up with the rejected noisy and ragged items of the later chunks."""
    k, h, w = 8, 496, 512
    clean = synth.layered_pair(4, h, w, k, seed=901)
    noisy = synth.layered_pair(4, h, w, k, seed=902, noise=2e-3)
    rt, rp = synth.ragged_pair_device(4, h, w, k, seed=903, device=cuda)
    yt = np.concatenate([clean[0], noisy[0], rt.cpu().numpy()])
    yp = np.concatenate([clean[1], noisy[1], rp.cpu().numpy()])
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    for max_pts in (None, 256):
        whole, _ = _evaluate(t, p, k, max_pts=max_pts)
        ref = whole.integers()
        assert ref["unsorted"][:4].tolist() == [0] * 4 and all(ref["unsorted"][4:] != 0)
        bound = suite.default_max_pts(w) if max_pts is None else max_pts
        per_item = k * 2 * bound * 4 * 2
        monkeypatch.setattr(suite, "CONTOUR_CHUNK_BYTES", 4 * per_item)
        assert len(yt) // (suite.CONTOUR_CHUNK_BYTES // per_item) >= 3
        res, _ = _evaluate(t, p, k, max_pts=max_pts)
        got = res.integers()
        if max_pts == 256:
            assert int(got["contour_n_pts"].max()) > 256          # the overflow retry ran
        for key, val in ref.items():
            if key == "contour_sum_dist":
                np.testing.assert_allclose(got[key], val, rtol=go.SUM_RTOL)
            else:
                assert np.array_equal(got[key], val), key
        go.check_suite(yt, yp, k, res)
        monkeypatch.undo()
