"""The geometry oracle itself (no GPU): its KD-tree distances equal the brute-force search, and its sawtooth pairs have
contours of exactly the requested length."""
import numpy as np
import pytest

from oracle import contours_oracle as co
from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

import geometry_oracle as go


def _pairs():
    rng = np.random.default_rng(7)
    for s in range(6):
        yield rng.random((24, 31)) < 0.3, rng.random((24, 31)) < 0.5
    yt, yp = synth.layered_pair(2, 96, 128, 5, seed=8, noise=2e-3)
    for i in range(2):
        for c in range(5):
            yield yt[i] == c, yp[i] == c


def test_kdtree_distances_equal_the_brute_force_search():
    n = 0
    for mt, mp in _pairs():
        for a, b in ((mt, mp), (mp, mt)):
            va, vb = co.all_crack_vertices(a), co.all_crack_vertices(b)
            if len(va) == 0 or len(vb) == 0:
                continue
            np.testing.assert_array_equal(go.nearest_sq(va, vb), co.directed_sq_distances(va, vb))
            n += 1
        try:
            vt, vp = co.first_contour_lattice(mt), co.first_contour_lattice(mp)
        except IndexError:
            continue
        np.testing.assert_array_equal(go.nearest_sq(vt, vp), co.directed_sq_distances(vt, vp))
    assert n >= 20


def test_contour_oracle_matches_the_label_map_oracle():
    yt, yp = synth.layered_pair(1, 64, 96, 4, seed=9, noise=5e-3)
    for c in range(4):
        r = go.contour_oracle(yt[0] == c, yp[0] == c)
        im = lo.contour_intermediates(yt[0] == c, yp[0] == c)
        assert (r is None) == (im is None)
        if r is None:
            continue
        assert r["n_pts"] == (len(im["verts_true"]), len(im["verts_pred"]))
        assert r[0] == go.order_stats(im["sq_pred_to_true"]) and r[1] == go.order_stats(im["sq_true_to_pred"])


@pytest.mark.parametrize("n_vertices", [65535, 65536, 65537])
@pytest.mark.parametrize("shift", [0, 1])
def test_sawtooth_pair_has_the_requested_vertex_count(n_vertices, shift):
    yt, yp = go.sawtooth_pair(128, 1024, n_vertices, shift)
    assert yt.shape == yp.shape == (1, 128, 1024) and yt.dtype == np.uint8
    assert len(co.first_contour_lattice(yt[0] == 0)) == n_vertices
    assert len(co.first_contour_lattice(yp[0] == 0)) == n_vertices
    assert (np.diff(yt[0].astype(np.int16), axis=0) >= 0).all()           # class order in every column
    assert np.array_equal(yp[0, shift:], yt[0, :128 - shift]) and not yp[0, :shift].any()


def test_sawtooth_pair_rejects_counts_that_do_not_fit():
    with pytest.raises(ValueError):
        go.sawtooth_pair(16, 64, 5000, 0)
    with pytest.raises(ValueError):
        go.sawtooth_pair(16, 64, 10, 0)
