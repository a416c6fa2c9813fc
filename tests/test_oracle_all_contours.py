"""CPU tier: the all-contour oracle equals what the restated find_contours gives with every contour concatenated."""
import numpy as np

from oracle import contours_oracle as co
from oracle import labelmap_oracle as lo
import all_contours_oracle as ao


def _rand_masks(seed, count=60):
    rng = np.random.default_rng(seed)
    for _ in range(count):
        h, w = rng.integers(2, 21, size=2)
        m = (rng.random((h, w)) < rng.uniform(0.1, 0.9)).astype(np.uint8)
        if rng.random() < 0.1:
            m[:] = rng.integers(0, 2)                 # empty or full: no contour at all
        yield m


def _brute_force_vertices(mask):
    """unique(concatenate(find_contours(mask, 0.5))) * 2, sorted by (row, col)."""
    cs = co.find_contours(mask, 0.5)
    if not cs:
        return np.zeros((0, 2), dtype=np.int64)
    return np.unique(np.concatenate([co.to_lattice(c) for c in cs]), axis=0)


def test_vertices_are_the_deduplicated_union_of_all_contours_in_raster_order():
    for m in _rand_masks(5):
        got = ao.all_vertices(m)
        ref = _brute_force_vertices(m)
        np.testing.assert_array_equal(got, ref)       # np.unique sorts rows lexicographically: raster order
        packed = ao.pack(got)
        assert np.all(np.diff(packed.astype(np.int64)) > 0)     # strictly increasing: each vertex once


def test_metrics_equal_brute_force_over_all_contours():
    masks = list(_rand_masks(6))
    for a, b in zip(masks[::2], masks[1::2]):
        h, w = min(a.shape[0], b.shape[0]), min(a.shape[1], b.shape[1])
        a, b = a[:h, :w], b[:h, :w]
        if h < 2 or w < 2:
            continue
        im = ao.all_contour_intermediates(a, b)
        vt, vp = _brute_force_vertices(a), _brute_force_vertices(b)
        if len(vt) == 0 or len(vp) == 0:
            assert im is None
            continue
        d1 = np.array([np.min(np.sqrt(np.sum((vt / 2.0 - p / 2.0) ** 2, axis=1))) for p in vp])
        d2 = np.array([np.min(np.sqrt(np.sum((vp / 2.0 - p / 2.0) ** 2, axis=1))) for p in vt])
        got = lo.contour_metrics_from_sq(im["sq_pred_to_true"], im["sq_true_to_pred"])
        assert got["hausdorff_distance"] == max(np.max(d1), np.max(d2))
        np.testing.assert_allclose(got["hausdorff_distance_95"], max(np.percentile(d1, 95), np.percentile(d2, 95)),
                                   rtol=1e-12)
        np.testing.assert_allclose(got["assd"], (np.mean(d1) + np.mean(d2)) / 2, rtol=1e-12)


def test_edt_distances_equal_brute_force():
    rng = np.random.default_rng(7)
    for _ in range(8):
        h, w = rng.integers(20, 70, size=2)
        a = rng.random((h, w)) < rng.uniform(0.02, 0.5)
        b = rng.random((h, w)) < rng.uniform(0.02, 0.5)
        vt, vp = ao.all_vertices(a), ao.all_vertices(b)
        np.testing.assert_array_equal(ao.edt_sq_distances(vt, vp, a.shape), co.directed_sq_distances(vt, vp))
        np.testing.assert_array_equal(ao.edt_sq_distances(vp, vt, a.shape), co.directed_sq_distances(vp, vt))


def test_single_closed_contour_is_contour_zero_without_its_repeat():
    m = np.zeros((12, 15), dtype=np.uint8)
    m[3:8, 4:11] = 1
    m[3, 6] = 0                 # a notch in the outline, still one closed contour
    first = co.first_contour_lattice(m)
    assert np.array_equal(first[0], first[-1])
    np.testing.assert_array_equal(ao.all_vertices(m), np.unique(first, axis=0))
    assert len(ao.all_vertices(m)) == len(first) - 1
