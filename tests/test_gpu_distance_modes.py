"""GPU exactness of the two vertex-list distance searches: the column-sorted search (the sorted source contour fits
shared memory) and the tiled box search (it does not) return, for every contour vertex, the exact squared distance to
the nearest vertex of the other contour -- pruning and tiling never change a result.  The reference is a host
nearest-neighbour search, independent of the GPU."""
import numpy as np
import pytest
import torch
from scipy.spatial import cKDTree

from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite, synth

pytestmark = pytest.mark.gpu


def _inputs(dev):
    yt, yp = synth.layered_pair(3, 200, 256, 6, seed=71, noise=0.002)
    yield "layered", torch.from_numpy(yt).to(dev), torch.from_numpy(yp).to(dev), 6
    yt, yp = synth.lesion_pair(3, 160, 160, 4, seed=72, single_blob_interior=False)
    yield "lesion", torch.from_numpy(yt).to(dev), torch.from_numpy(yp).to(dev), 4
    # ragged predictions at W = 1024: contours longer than one 2048-vertex tile of the tiled search
    yt, yp = synth.ragged_pair_device(2, 256, 1024, 6, seed=73, device=dev)
    yield "ragged", yt, yp, 6


def _lattice(v):
    """Doubled-lattice (y2, x2) of packed vertices y2 << 16 | x2."""
    v = v.astype(np.int64)
    return np.stack([v >> 16, v & 0xffff], axis=1)


def _nearest_sq(src, qry):
    """Exact squared distance from every query vertex to its nearest source vertex (integers: the tree only picks
    the index)."""
    _, idx = cKDTree(src).query(qry)
    d = qry - src[idx]
    return (d * d).sum(axis=1)


def _stats(d):
    """max, the two neighbours of numpy's linear 95th percentile, sum of sqrt(d / 4)."""
    s = np.sort(d)
    lo = int(np.floor((len(s) - 1) * 0.95))
    return int(s[-1]), [int(s[lo]), int(s[min(lo + 1, len(s) - 1)])], float(np.sqrt(s / 4.0).sum())


# max_pts -> the search it selects: 8192 sorted vertices (~139 KB at W = 1024) fit shared memory, 16384 (~270 KB) do not
PATHS = [(8192, "distance_column_kernel"), (16384, "distance_search_kernel")]


def test_all_modes_agree(cuda):
    for max_pts, kernel in PATHS:
        _check_path(cuda, max_pts, kernel)


def _check_path(cuda, max_pts, kernel):
    for name, yt, yp, k in _inputs(cuda):
        with _lib.kernel_profile() as prof:
            ct = suite.contour_pass(yt, yp, k, max_pts=max_pts, return_vertices=True, return_sq=True)
            torch.cuda.synchronize()
        assert kernel in prof.kernels, (name, sorted(prof.kernels))
        n = ct.n_pts.cpu().numpy().view(np.uint32)
        verts = ct.verts.cpu().numpy().view(np.uint32)
        sq = ct.sq.cpu().numpy().view(np.uint32)
        max_sq = ct.max_sq.cpu().numpy().view(np.uint32)
        p95_sq = ct.p95_sq.cpu().numpy().view(np.uint32)
        sum_dist = ct.sum_dist.cpu().numpy()
        if name == "ragged":
            assert n.max() > 2048, n.max()
        for i in range(n.shape[0]):
            for c in range(k):
                pts = [_lattice(verts[i, c, m, :n[i, c, m]]) for m in range(2)]
                for d in range(2):      # direction 0: queries = pred vertices (map 1), sources = true vertices (map 0)
                    where = (name, i, c, d)
                    if len(pts[0]) == 0 or len(pts[1]) == 0:
                        assert max_sq[i, c, d] == 0 and p95_sq[i, c, d].tolist() == [0, 0] and sum_dist[i, c, d] == 0, where
                        continue
                    ref = _nearest_sq(pts[d], pts[1 - d])
                    np.testing.assert_array_equal(sq[i, c, d, :len(ref)], ref, err_msg=str(where))
                    vmax, p95, dsum = _stats(ref)
                    assert max_sq[i, c, d] == vmax and p95_sq[i, c, d].tolist() == p95, where
                    np.testing.assert_allclose(sum_dist[i, c, d], dsum, rtol=1e-12, err_msg=str(where))
        # without return_sq the search counts the distances instead of storing them: same integers, sums equal up to
        # the order of the float64 additions
        with _lib.kernel_profile() as prof:
            ct2 = suite.contour_pass(yt, yp, k, max_pts=max_pts)
            torch.cuda.synchronize()
        assert kernel in prof.kernels, (name, sorted(prof.kernels))
        assert torch.equal(ct2.max_sq, ct.max_sq) and torch.equal(ct2.p95_sq, ct.p95_sq), name
        np.testing.assert_allclose(ct2.sum_dist.cpu().numpy(), sum_dist, rtol=1e-12)
