"""GPU: per-sector layer thickness of OCT volumes (``suite.sector_thickness``, ``octm_sector_thickness_i32``) bit for bit
against ``tests/sector_thickness_oracle.py``, on the label-pass kernels each shape takes: the TMA column-strip kernel
(Duke DME, K = 8, W % 16 == 0), the warp-per-strip kernel (HC-MS, K = 10) and the byte-wise generic kernel (odd W)."""
import numpy as np
import pytest

import sector_thickness_oracle as sto
from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, synth

pytestmark = pytest.mark.gpu
DUKE_SP = (0.1185, 0.00387, 0.00772)       # mm: B-scans, rows, columns
HCMS_SP = (0.1229, 0.00387, 0.00583)
NARROW_SP = (0.12, 0.004, 0.02)            # 301 columns span 6 mm


def _dev(cuda, *arrs):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).to(cuda) for a in arrs)


def _volumes(kind, v, b, h, w, k, seed):
    n = v * b
    if kind == "layered":
        yt, yp = synth.layered_pair(n, h, w, k, seed=seed)
    elif kind == "noisy":
        yt, yp = synth.layered_pair(n, h, w, k, seed=seed, noise=0.02)
    elif kind == "ragged":
        import torch
        yt, yp = (t.cpu().numpy() for t in synth.ragged_pair_device(n, h, w, k, seed=seed, device=torch.device("cuda", 0)))
    elif kind == "random":
        yt, yp = synth.random_pair(n, h, w, k, seed=seed)
    else:
        yt, yp = synth.lesion_pair(n, h, w, k, seed=seed, single_blob_interior=False)
    return yt.reshape(v, b, h, w), yp.reshape(v, b, h, w)


def _expected(yt, yp, k, groups, spacing, centers, radii=derive.ETDRS_RADII):
    v, b, _, w = yt.shape
    regions = np.stack([derive.etdrs_regions(b, w, spacing, c, radii) for c in centers])
    return sto.sector_sums(yt, yp, k, groups, regions, len(derive.ETDRS_SECTORS))


def _check(cuda, yt, yp, k, spacing, center=None, classes=None, radii=derive.ETDRS_RADII):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    dt, dp = _dev(cuda, yt, yp)
    out = suite.sector_thickness(dt, dp, k, spacing, center=center, classes=classes, radii=radii, maps=True)
    ints = out.integers()
    groups = derive.sector_groups(classes, k)
    if yt.ndim == 3:                         # [B, H, W]: one volume
        yt, yp = yt[None], yp[None]
    centers = derive.sector_centers(center, yt.shape[0], yt.shape[1], yt.shape[3])
    want_sums, want_maps = _expected(yt, yp, k, groups, spacing, centers, radii)
    assert ints["sums"].dtype == np.int64 and ints["maps"].dtype == np.int32
    assert np.array_equal(ints["sums"], want_sums)
    assert np.array_equal(ints["maps"], want_maps)
    return out, want_sums


KINDS = ("layered", "noisy", "ragged", "random", "lesion")
SHAPES = {"duke": (2, 61, 496, 768, 8, DUKE_SP, 1), "hcms": (2, 49, 496, 1024, 10, HCMS_SP, 2),
          "generic": (2, 9, 120, 301, 6, NARROW_SP, 0)}


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_bit_exact_against_oracle(cuda, shape, kind):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    v, b, h, w, k, sp, path = SHAPES[shape]
    if kind != "layered":
        b = min(b, 7)                        # the full B-scan count once per shape, on the layered maps
    assert _lib.load().octm_label_pass_path(h, w, k, 0, 0) == path
    yt, yp = _volumes(kind, v, b, h, w, k, seed=100 * list(SHAPES).index(shape) + KINDS.index(kind))
    out, want = _check(cuda, yt, yp, k, sp)
    m = out.metrics()
    assert np.array_equal(m["n_ascans"], want[..., 0])
    ref = derive.sector_thickness(want, sp)
    for key in ref:
        assert np.array_equal(m[key], ref[key], equal_nan=True), key


def test_mixed_centres_in_one_call(cuda):
    v, b, h, w, k = 4, 13, 160, 256, 8
    yt, yp = _volumes("noisy", v, b, h, w, k, seed=31)
    sp = (0.4, 0.004, 0.025)                 # 5.2 mm by 6.4 mm
    centers = np.array([[6.0, 127.5], [3.25, 40.0], [12.0, 255.0], [-4.0, 300.0]])   # the last is partly outside
    out, want = _check(cuda, yt, yp, k, sp, center=centers)
    assert want[3, :, 0, 0].sum() == 0 and want[3, :, :, 0].sum() > 0      # no centre subfield, some outer ring
    _check(cuda, yt, yp, k, sp, center=(5.5, 100.25))                       # one pair for every volume


def test_single_bscan_volumes(cuda):
    yt, yp = _volumes("layered", 3, 1, 96, 200, 5, seed=8)
    _check(cuda, yt, yp, 5, (1.0, 0.004, 0.03))
    _check(cuda, yt[:, 0], yp[:, 0], 5, (1.0, 0.004, 0.03))                 # [B, H, W] is one volume


def test_groups(cuda):
    yt, yp = _volumes("noisy", 2, 11, 200, 384, 8, seed=12)
    classes = [(1, 7), 0, 7, (2, 4), (0, 7), (6, 7)]
    out, want = _check(cuda, yt, yp, 8, (0.3, 0.004, 0.016), classes=classes)
    assert out.groups == ((1, 7), (0, 0), (7, 7), (2, 4), (0, 7), (6, 7))
    assert np.all(out.integers()["maps"][:, :, :, 4] == 200)                 # all classes: the whole A-scan
    _check(cuda, yt, yp, 8, (0.3, 0.004, 0.016), classes=list(range(8)) * 2)  # 16 groups


def test_tall_maps_reduce_in_64_bits(cuda):
    """Tall maps: (t - p)^2 of about 11880^2 summed over 32 lanes of one region exceeds 2^32."""
    rng = np.random.default_rng(3)
    v, b, h, w, k = 1, 2, 12000, 37, 3
    yt = np.zeros((v, b, h, w), np.uint8)
    yp = np.zeros((v, b, h, w), np.uint8)
    yt[..., 11900:, :] = 1
    yp[..., 10:, :] = 1
    yp[..., 11990:, :] = 2
    yt[..., 50, :] = rng.integers(0, k, size=(v, b, w))
    out, want = _check(cuda, yt, yp, k, (1.0, 0.001, 1.0), radii=(1e5, 2e5, 3e5))
    assert want[0, 1, 0, 4] >= 32 * 11870 ** 2 > 2 ** 32


def test_bool_maps(cuda):
    rng = np.random.default_rng(4)
    yt = rng.random((2, 5, 40, 64)) < 0.4
    yp = rng.random((2, 5, 40, 64)) < 0.4
    _check(cuda, yt, yp, 2, (0.5, 0.01, 0.1), classes=[1, (0, 1)])


def test_matches_the_label_pass_thickness(cuda):
    """Single-class groups and one region holding every A-scan of a one-B-scan volume: sum |t - p| is the label pass's
    thick_absdiff of that B-scan."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    for kind, (h, w, k) in (("ragged", (496, 512, 8)), ("noisy", (496, 1024, 10)), ("lesion", (77, 301, 4))):
        yt, yp = _volumes(kind, 6, 1, h, w, k, seed=19)
        dt, dp = _dev(cuda, yt, yp)
        out = suite.sector_thickness(dt, dp, k, (1.0, 1.0, 1.0), radii=(1e9, 2e9, 3e9))
        sums = out.integers()["sums"]
        assert np.all(sums[:, :, 1:, 0] == 0) and np.all(sums[:, :, 0, 0] == w)
        lp = suite.label_pass(dt[:, 0], dp[:, 0], k, counts=True, columns=True)
        assert np.array_equal(sums[:, :, 0, 3], lp.thick_absdiff.cpu().numpy()), kind
        for i in range(6):
            ref = lo.score_bscan_fast(yt[i, 0], yp[i, 0], k)
            assert np.array_equal(sums[i, :, 0, 1], ref["thickness_true"].sum(1))


def test_label_out_of_range_raises(cuda):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    for h, w, k in ((496, 768, 8), (496, 1024, 10), (50, 301, 4)):
        yt, yp = _volumes("layered", 2, 3, h, w, k, seed=2)
        yp[1, 2, 10, 5] = 255
        dt, dp = _dev(cuda, yt, yp)
        out = suite.sector_thickness(dt, dp, k, (0.1, 0.004, 0.01))
        with pytest.raises(ValueError, match="label >= num_classes"):
            out.integers()
        with pytest.raises(ValueError, match="label >= num_classes"):
            out.metrics()
        assert out.bad_label_items() == 1


def test_repeated_calls_are_bit_identical(cuda):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = _volumes("random", 3, 8, 128, 512, 8, seed=5)
    dt, dp = _dev(cuda, yt, yp)
    first = suite.sector_thickness(dt, dp, 8, (0.2, 0.004, 0.012), maps=True).integers()
    for _ in range(3):
        again = suite.sector_thickness(dt, dp, 8, (0.2, 0.004, 0.012), maps=True).integers()
        for key in first:
            assert np.array_equal(again[key], first[key]), key


def test_single_rank_totals_on_the_device(cuda):
    """dist.sector_thickness_totals with world 1 takes the device result as it is."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = _volumes("noisy", 3, 5, 64, 128, 4, seed=6)
    dt, dp = _dev(cuda, yt, yp)
    out = suite.sector_thickness(dt, dp, 4, (0.5, 0.004, 0.04))
    tot = odist.sector_thickness_totals(out, 1, 0, 3)
    assert np.array_equal(tot["sums"], out.integers()["sums"])
    per = out.metrics()
    summ = derive.sector_thickness_summary(per)
    for key in summ:
        assert np.array_equal(tot["summary"][key], summ[key], equal_nan=True), key


def test_empty_batch(cuda):
    """No volume at all: every output is empty and reading it works, as for a rank that holds no shard."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    y = torch.zeros((0, 7, 64, 128), dtype=torch.uint8, device=cuda)
    out = suite.sector_thickness(y, y, 4, (0.5, 0.004, 0.04), maps=True)
    ints = out.integers()
    assert ints["sums"].shape == (0, 4, 9, 5) and ints["maps"].shape == (0, 7, 2, 4, 128)
    assert out.bad_label_items() == 0
    assert out.metrics()["thickness_mae"].shape == (0, 4, 9)
    assert odist.sector_thickness_totals(out, 1, 0, 0)["sums"].shape == (0, 4, 9, 5)


def test_groups_sharing_boundary_rows(cuda):
    """Consecutive groups where one starts at the class after the previous one ends reuse that boundary row."""
    yt, yp = _volumes("ragged", 2, 5, 160, 256, 8, seed=23)
    _check(cuda, yt, yp, 8, (0.5, 0.004, 0.025), classes=[0, 1, (2, 7), 0, (0, 3), (4, 5), 6, (7, 7), (3, 7)])
