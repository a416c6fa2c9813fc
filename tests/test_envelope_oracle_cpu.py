"""The fast envelope oracles (no GPU) equal the brute-force ones bit for bit: all-contour squared distances, squared
distances at a pixel spacing (OCT, 30:1 and dyadic, in both contour modes), and surface Dice counts, tolerance ties
included."""
import numpy as np
import pytest

from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, synth

import all_contours_oracle as ao
import envelope_oracle as eo
import spacing_2d_oracle as so
import surface_dice_oracle as sdo

SPACINGS = {"oct": (0.0039, 0.0117), "rows30": (30.0, 1.0), "cols30": (1.0, 30.0), "dyadic": (0.5, 2.0)}


def _items():
    rng = np.random.default_rng(17)
    for _ in range(3):
        yield "random", (rng.random((19, 27)) < 0.4).astype(np.uint8), (rng.random((19, 27)) < 0.5).astype(np.uint8), 2
    yt, yp = synth.layered_pair(2, 40, 64, 5, seed=18, noise=0.02)
    for i in range(2):
        yield "layered", yt[i], yp[i], 5
    yt, yp = synth.lesion_pair(2, 48, 56, 3, seed=19, single_blob_interior=False)
    for i in range(2):
        yield "lesion", yt[i], yp[i], 3


def test_all_contour_distances_equal_the_brute_force_search():
    n = 0
    for _, yt, yp, k in _items():
        for c, (vt, vp, d) in enumerate(eo.contours(yt, yp, k, "all")):
            assert np.array_equal(vt, ao.all_vertices(yt == c)) and np.array_equal(vp, ao.all_vertices(yp == c))
            if d is None:
                continue
            assert d[0].dtype == np.int64
            np.testing.assert_array_equal(d[0], ao.sq_distances(vt, vp, yt.shape))
            np.testing.assert_array_equal(d[1], ao.sq_distances(vp, vt, yt.shape))
            n += 1
    assert n >= 15


@pytest.mark.parametrize("mode", ["all", "first"])
@pytest.mark.parametrize("spacing", list(SPACINGS))
def test_spacing_distances_equal_the_brute_force_search(spacing, mode):
    sp = SPACINGS[spacing]
    n = 0
    for _, yt, yp, k in _items():
        for c, (vt, vp, d) in enumerate(eo.contours(yt, yp, k, mode, sp)):
            if d is None:
                assert so.intermediates(yt == c, yp == c, sp, mode) is None
                continue
            ref = so.intermediates(yt == c, yp == c, sp, mode)
            assert np.array_equal(d[0], ref["sq_pred_to_true"]) and np.array_equal(d[1], ref["sq_true_to_pred"])
            n += 1
    assert n >= 15


def test_spacing_distances_on_many_ties():
    """Equidistant candidates everywhere: a lattice against its own shift at spacings where many q coincide."""
    y, x = np.mgrid[0:40:2, 1:60:2]
    src = np.stack([y.ravel(), x.ravel()], axis=1)
    qry = src + np.array([1, 1])
    for sp in SPACINGS.values():
        np.testing.assert_array_equal(eo.spacing_d2(src, qry, sp), so.squared_distances(src, qry, sp))


def test_surface_counts_equal_the_brute_force_oracles():
    taus = (0.0, 1.0, np.sqrt(5.0) / 2, 8.0)
    for _, yt, yp, k in _items():
        ns, nw = eo.surface_counts(yt, yp, k, taus)
        for c in range(k):
            rs, rw = sdo.mask_counts(yt == c, yp == c, taus)
            assert np.array_equal(ns[c], rs) and np.array_equal(nw[c], rw), c


@pytest.mark.parametrize("spacing", list(SPACINGS))
def test_surface_counts_at_a_spacing_with_tolerance_ties(spacing):
    """Tolerances equal to distances that occur (exact at the dyadic spacing), the largest tolerance allowed, and 0."""
    sp = SPACINGS[spacing]
    items = list(_items())
    occurring = np.unique(np.concatenate([d[0] for _, yt, yp, k in items for _, _, d in eo.contours(yt, yp, k, "all", sp)
                                          if d is not None]))
    dist = np.sqrt(occurring / 4.0)
    lim = derive.surface_dice_spacing_limit(sp)
    ties = tuple(float(v) for v in dist[(dist > 0) & (dist <= lim)][:2]) + (lim, 0.0)
    assert len(ties) == 4
    for _, yt, yp, k in items:
        ns, nw = eo.surface_counts(yt, yp, k, ties, sp)
        for c in range(k):
            rs, rw = so.surface_dice_counts(yt == c, yp == c, sp, ties)
            assert tuple(ns[c]) == rs and np.array_equal(nw[c], rw), c


def test_all_contour_distances_at_8192_columns_equal_the_distance_transform():
    """At the envelope the brute-force search is out of reach; the EDT of the doubled lattice is the exact check."""
    yt, yp = synth.layered_pair(1, 48, 8192, 4, seed=20, noise=2e-3)
    ref = eo.contours(yt[0], yp[0], 4, "all")
    assert max(len(vt) for vt, _, _ in ref) > 8192
    for vt, vp, d in ref:
        np.testing.assert_array_equal(d[0], ao.edt_sq_distances(vt, vp, yt.shape[1:]))
        np.testing.assert_array_equal(d[1], ao.edt_sq_distances(vp, vt, yt.shape[1:]))
