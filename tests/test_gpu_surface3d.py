"""GPU parity: 3-D surface distances (exact separable EDT) against the scipy oracle: every squared-distance statistic
bit-exact (count, max, the two order statistics of the 95th percentile), distance sums to 1e-12 relative, hd bit-exact,
hd95 / assd within 1e-6 relative.

Each case asserts on its own inputs that it reaches the route it is named for.  The routes of csrc/edt3d.cu:
  * near-field path: D2 % 16 == 0 and both volumes 16-byte aligned; a unit whose query voxels are all closer than
    NEAR_CAP is settled there, any other unit ("overflowing") is redone by the general kernels;
  * general path, pass 1: the vectorised kernel when D2 % 16 == 0 and the unit's SOURCE volume is 16-byte aligned,
    the byte-wise kernel otherwise; pass 3 counts squared distances below SMEM_BINS in shared memory, the rest in
    global bins;
  * passes 2 and 3 keep stacks of MAX_LINE entries per thread.
"""
import numpy as np
import pytest

from oracle import surface3d_oracle as so
from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

pytestmark = pytest.mark.gpu
RTOL = 1e-6
NEAR_CAP = 121          # (kNearR + 1)^2 in edt3d.cu
SMEM_BINS = 8192        # kSmemBins
MAX_LINE = 2048         # kMaxLine
KEYS = ("sq_pred_to_true", "sq_true_to_pred")       # direction 0, direction 1


def _to(cuda, *vols):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(v)).to(cuda) for v in vols)


def _misaligned(t):
    """The same contents at an odd address: a contiguous view one byte into a fresh buffer (kept as is by the suite)."""
    import torch
    buf = torch.empty(t.numel() + 1, dtype=torch.uint8, device=t.device)
    v = buf[1:].view(t.shape).copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 2 == 1
    return v


def _aligned(*ts):
    return all(t.data_ptr() % 16 == 0 for t in ts)


def _check(vt, vp, k, cuda, vols=None):
    """Run the kernels on (vt, vp), or on the device tensors ``vols`` holding the same contents, and compare every
    output of every class and direction with the oracle.  Returns (outputs, {class: oracle result})."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    ints = suite.surface_distance_3d(*(vols if vols is not None else _to(cuda, vt, vp)), k)
    m = suite.surface_metrics_3d(ints)
    n_pts = ints["n_pts"].cpu().numpy().view(np.uint32)
    max_sq = ints["max_sq"].cpu().numpy().view(np.uint32)
    p95 = ints["p95_sq"].cpu().numpy().view(np.uint32)
    sums = ints["sum_dist"].cpu().numpy()
    refs = {}
    for c in range(k):
        ref = refs[c] = so.class_metrics(vt, vp, c)
        if ref["sq_pred_to_true"] is None:
            assert not (n_pts[c].any() or max_sq[c].any() or p95[c].any() or sums[c].any()), c
            assert np.isnan(m["hausdorff_distance"][c])
            continue
        for d, key in enumerate(KEYS):
            s = np.sort(ref[key])
            n = len(s)
            lo = int(np.floor((n - 1) * 0.95))
            assert n_pts[c, 1 - d] == n, (c, d)
            assert max_sq[c, d] == s[-1], (c, d, int(max_sq[c, d]), int(s[-1]))
            assert tuple(p95[c, d]) == (s[lo], s[min(lo + 1, n - 1)]), (c, d, tuple(p95[c, d]))
            np.testing.assert_allclose(sums[c, d], np.sqrt(s.astype(np.float64)).sum(), rtol=1e-12,
                                       err_msg=f"sum_dist class {c} direction {d}")
        assert m["hausdorff_distance"][c] == ref["hausdorff_distance"], c                  # bit-exact
        for name in ("hausdorff_distance_95", "assd"):
            np.testing.assert_allclose(m[name][c], ref[name], rtol=RTOL, atol=0, err_msg=f"{name} class {c}")
    return ints, refs


def _check_alignments(vt, vp, k, cuda):
    """D2 % 16 == 0 volumes three ways: both aligned (near-field path first); y_pred at an odd address (no near-field
    path, direction 0 reads the aligned y_true with the vectorised pass 1, direction 1 the odd y_pred byte-wise); both
    at odd addresses (every unit byte-wise on the general path).  All must match the oracle and each other exactly."""
    import torch
    assert vt.shape[2] % 16 == 0
    t, p = _to(cuda, vt, vp)
    assert _aligned(t, p)
    ref, refs = _check(vt, vp, k, cuda, vols=(t, p))
    for vols in ((t, _misaligned(p)), (_misaligned(t), _misaligned(p))):
        got, _ = _check(vt, vp, k, cuda, vols=vols)
        for key in ref:
            assert torch.equal(got[key], ref[key]), key
    return refs


def _mixed_volume():
    """Class 1 near, class 2 with an extra far island in the prediction (its direction 0 overflows), class 3 exactly
    at the cap."""
    vt = np.zeros((40, 36, 32), np.uint8)
    vp = np.zeros((40, 36, 32), np.uint8)
    vt[5:20, 4:30, 3:29] = 1                           # class 1: two boxes one or two voxels apart (near)
    vp[6:21, 5:30, 2:28] = 1
    vt[25:38, 2:10, 2:12] = 2                          # class 2: the prediction has an extra island 20 voxels away (far)
    vp[25:38, 2:10, 2:12] = 2
    vp[26:30, 30:34, 24:30] = 2
    vt[22, 20:24, 16] = 3                              # class 3: exactly at the cap: distance 11 along one axis
    vp[22, 20:24, 27] = 3
    return vt, vp


def test_layered_volume(cuda):
    vt, vp = synth.layered_volume_pair(48, 40, 24, 5, seed=51)
    _check(vt, vp, 5, cuda)


def test_random_blobs_and_missing_class(cuda):
    rng = np.random.default_rng(52)
    vt = (rng.random((20, 33, 17)) < 0.3).astype(np.uint8) + (rng.random((20, 33, 17)) < 0.1).astype(np.uint8)
    vp = (rng.random((20, 33, 17)) < 0.3).astype(np.uint8) + (rng.random((20, 33, 17)) < 0.1).astype(np.uint8)
    vp[vp == 2] = 1                                    # class 2 absent from the prediction -> undefined
    _check(vt, vp, 4, cuda)                            # class 3 absent from both


def test_vectorised_first_pass_shapes(cuda):
    """D2 a multiple of 16: the 16-voxel first pass (borders, thin sheets, runs crossing group boundaries)"""
    rng = np.random.default_rng(54)
    for shape in ((12, 9, 32), (7, 11, 48), (5, 6, 16)):
        vt = (rng.random(shape) < 0.5).astype(np.uint8)
        vp = (rng.random(shape) < 0.5).astype(np.uint8)
        vt[:, :, 10:20] = 1                                # long run along the contiguous axis
        _check(vt, vp, 2, cuda)
    vt, vp = synth.layered_volume_pair(40, 24, 32, 4, seed=55)
    _check(vt, vp, 4, cuda)


def test_far_apart_and_border_touching(cuda):
    vt = np.zeros((120, 80, 12), np.uint8)
    vp = np.zeros((120, 80, 12), np.uint8)
    vt[0:6, 0:5, :] = 1                                # touches four faces of the volume
    vp[100:120, 70:80, 3:9] = 1                        # far corner: squared distances up to 114^2 + 75^2 = 18621
    _, refs = _check(vt, vp, 2, cuda)
    assert refs[1]["sq_pred_to_true"].max() >= SMEM_BINS               # global bins


# one class per single-voxel pair: (y_true voxel, y_pred voxel, squared distance)
FAR_PAIRS = {1: ((2, 2, 2), (92, 2, 2), 8100),            # 90^2: the last shared-memory bins below the boundary
             2: ((2, 5, 5), (66, 69, 5), 8192),           # 64^2 + 64^2: the first global bin
             3: ((5, 2, 10), (69, 66, 11), 8193),         # 64^2 + 64^2 + 1
             4: ((0, 0, 20), (159, 71, 31), 30443)}       # 159^2 + 71^2 + 11^2: 174 voxels apart


def test_far_field_and_the_global_histogram(cuda):
    """Single query voxels on both sides of the shared / global bin boundary of pass 3 (max_sq and both p95 entries
    equal the one distance), then one unit with many query voxels on both sides of it spread over the whole volume."""
    for d2 in (32, 33):                 # near-field attempt overflows, then the vectorised pass 1; the byte-wise pass 1
        vt = np.zeros((160, 72, d2), np.uint8)
        vp = np.zeros((160, 72, d2), np.uint8)
        for c, (a, b, _) in FAR_PAIRS.items():
            vt[a] = c
            vp[b] = c
        t, p = _to(cuda, vt, vp)
        assert _aligned(t, p)
        _, refs = _check(vt, vp, 5, cuda, vols=(t, p))
        for c, (_, _, want) in FAR_PAIRS.items():
            for key in KEYS:
                assert refs[c][key].tolist() == [want], (c, key)
    # a source blob at one end, ~1100 single query voxels through the rest of a 300-voxel-long volume
    rng = np.random.default_rng(58)
    vt = np.zeros((300, 40, 48), np.uint8)
    vt[0:6, 10:30, 12:36] = 1
    vp = np.zeros((300, 40, 48), np.uint8)
    vp[10:] = rng.random((290, 40, 48)) < 0.002
    _, refs = _check(vt, vp, 2, cuda)
    s = refs[1]["sq_pred_to_true"]
    assert (s < SMEM_BINS).sum() >= 100 and (s >= SMEM_BINS).sum() >= 100


def test_long_lines(cuda):
    """Lines of MAX_LINE voxels along D0 (pass-3 stacks) and D1 (pass-2 stacks), and of 4095 / 4096 along D2 (pass-1
    distances).  Class 1: sparse random surface in both volumes.  Class 2: a whole line along the long axis in one corner
    of y_true and in the opposite corner of y_pred; every voxel of it is surface and equally far from the other, so each
    envelope over such lines keeps every site and its stack fills to the line length.  Class 3: one voxel at each end of
    the long axis, in opposite corners: the volume's diagonal."""
    rng = np.random.default_rng(59)
    for shape in ((2048, 3, 16), (3, 2048, 16), (2048, 2, 17), (2, 3, 4096), (2, 3, 4095)):
        axis = int(np.argmax(shape))
        L = shape[axis]
        vt = (rng.random(shape) < 0.001).astype(np.uint8)
        vp = (rng.random(shape) < 0.001).astype(np.uint8)
        lt, lp = [0, 0, 0], [-1, -1, -1]
        lt[axis] = lp[axis] = slice(None)
        vt[tuple(lt)] = 2
        vp[tuple(lp)] = 2
        et, ep = [-1, -1, -1], [0, 0, 0]               # corners away from y_true's / y_pred's class-2 line
        et[axis], ep[axis] = 0, -1
        vt[tuple(et)] = 3
        vp[tuple(ep)] = 3
        _, refs = _check(vt, vp, 4, cuda)
        across = sum((s - 1) ** 2 for i, s in enumerate(shape) if i != axis)
        assert L in (MAX_LINE, 4095, 4096) and (L - 1) ** 2 + across >= NEAR_CAP
        assert axis == 2 or across >= NEAR_CAP         # the class-2 units whose stacks fill leave the near field
        for key in KEYS:
            assert refs[2][key].tolist() == [across] * L, key
            assert refs[3][key].tolist() == [(L - 1) ** 2 + across], key
        assert len(refs[1]["sq_pred_to_true"]) >= 3


def test_every_class_voxel_is_surface(cuda):
    """Volumes one voxel thick on two or three axes: every voxel of every class is surface."""
    rng = np.random.default_rng(60)
    for shape in ((1, 1, 1), (1, 1, 40), (40, 1, 1), (1, 30, 16)):
        vt = rng.integers(0, 3, shape, dtype=np.uint8)
        vp = rng.integers(0, 3, shape, dtype=np.uint8)
        if shape == (1, 1, 1):
            vt[:] = vp[:] = 1
        for v in (vt, vp):
            for c in range(3):
                assert np.array_equal(so.surface(v == c), v == c)
        _check(vt, vp, 3, cuda)


def test_misaligned_volumes(cuda):
    """The general path on units that never tried the near-field path, and one call mixing both pass-1 kernels."""
    refs = _check_alignments(*_mixed_volume(), 4, cuda)
    assert refs[1]["sq_pred_to_true"].max() < NEAR_CAP <= refs[2]["sq_pred_to_true"].max()
    vt = np.zeros((160, 72, 32), np.uint8)
    vp = np.zeros((160, 72, 32), np.uint8)
    for c, (a, b, _) in FAR_PAIRS.items():
        vt[a] = c
        vp[b] = c
    _check_alignments(vt, vp, 5, cuda)
    _check_alignments(*synth.layered_volume_pair(40, 24, 32, 4, seed=55), 4, cuda)


HIGH_CLASSES = (1, 127, 128, 254, 255)


def test_class_values_up_to_255(cuda):
    """K = 256.  Each of HIGH_CLASSES once with a near-field unit (direction 0) and an overflowing one (direction 1);
    then uniform random labels in 0..255, aligned (a few units overflow) and at odd addresses (all 512 units on the
    general path)."""
    vt = np.zeros((48, 32, 32), np.uint8)
    vp = np.zeros((48, 32, 32), np.uint8)
    for j, c in enumerate(HIGH_CLASSES):
        b = 9 * j + 1
        vt[b:b + 6, 2:8, 2:8] = c
        vp[b:b + 6, 2:8, 3:9] = c                      # one voxel along D2: direction 0 stays in the near field
        vt[b + 3, 28, 28] = c                          # an island of y_true 29 voxels from y_pred: direction 1 overflows
    t, p = _to(cuda, vt, vp)
    assert _aligned(t, p)
    _, refs = _check(vt, vp, 256, cuda, vols=(t, p))
    for c in HIGH_CLASSES:
        assert refs[c]["sq_pred_to_true"].max() < NEAR_CAP <= refs[c]["sq_true_to_pred"].max(), c
    rng = np.random.default_rng(57)
    vt = rng.integers(0, 256, (16, 16, 32), dtype=np.uint8)
    vp = rng.integers(0, 256, (16, 16, 32), dtype=np.uint8)
    refs = _check_alignments(vt, vp, 256, cuda)
    far = [refs[c][key].max() >= NEAR_CAP for c in range(256) for key in KEYS]
    assert 0 < sum(far) < len(far) == 512


def test_class_255_on_the_last_d2_face(cuda):
    """The vectorised pass 1 reads past the end of each line; that padding must not count as a class-255 neighbour,
    or the class-255 voxels on the last D2 face whose other neighbours are 255 lose their surface mark."""
    vt = np.zeros((8, 8, 32), np.uint8)
    vt[2:6, 2:6, 20:32] = 255                          # touches the last D2 face, interior in D0 / D1
    vp = vt.copy()
    vp[1, 1, 0] = 255                                  # island 20 voxels from y_true's surface: direction 0 overflows
    refs = _check_alignments(vt, vp, 256, cuda)        # aligned first: direction 0 reads y_true with the vectorised pass
    assert refs[255]["sq_pred_to_true"].max() >= NEAR_CAP


def test_unit_ranges_add_up(cuda):
    """Disjoint unit ranges add up to the full call; each single unit writes its own entries only; repeated calls are
    bit-identical (sum_dist included: the select kernel sums in a fixed order); bool volumes equal uint8 0/1 ones."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    mixed = _mixed_volume()
    for vt, vp in (synth.layered_volume_pair(32, 24, 16, 4, seed=53), mixed):
        full, _ = _check(vt, vp, 4, cuda)
        t, p = _to(cuda, vt, vp)
        a = suite.surface_distance_3d(t, p, 4, units=(0, 3))
        b = suite.surface_distance_3d(t, p, 4, units=(3, 8))
        for key in full:
            assert torch.equal(a[key] + b[key], full[key]), key
        for u in range(8):
            c, d = divmod(u, 2)
            one = suite.surface_distance_3d(t, p, 4, units=(u, u + 1))
            for key, at in (("n_pts", (c, 1 - d)), ("max_sq", (c, d)), ("p95_sq", (c, d)), ("sum_dist", (c, d))):
                mine = torch.zeros(full[key].shape, dtype=torch.bool, device=cuda)
                mine[at] = True
                assert torch.equal(one[key][mine], full[key][mine]), (u, key)
                assert not one[key][~mine].any(), (u, key)
        again = suite.surface_distance_3d(t, p, 4)
        for key in full:
            assert torch.equal(again[key], full[key]), key
    vt, vp = mixed
    assert so.class_metrics(vt, vp, 2)["sq_pred_to_true"].max() >= NEAR_CAP
    t, p = _to(cuda, vt == 2, vp == 2)
    assert t.dtype == torch.bool
    as_bool = suite.surface_distance_3d(t, p, 2)
    as_u8 = suite.surface_distance_3d(t.to(torch.uint8), p.to(torch.uint8), 2)
    for key in as_u8:
        assert torch.equal(as_bool[key], as_u8[key]), key


def test_near_field_path_and_its_overflow(cuda):
    """D2 % 16 == 0 takes the capped windowed transform (exact below (R+1)^2 = 121); a unit with a single query voxel at
    or beyond the cap must be redone by the general kernels, while the other units of the same call keep the fast result."""
    rng = np.random.default_rng(56)
    _, refs = _check(*_mixed_volume(), 4, cuda)
    assert refs[1]["sq_pred_to_true"].max() < NEAR_CAP <= refs[2]["sq_pred_to_true"].max()
    assert refs[3]["sq_pred_to_true"].max() == NEAR_CAP
    # distances 10 (below the cap) and 11 (at the cap) along each axis in turn
    for axis in range(3):
        for gap in (10, 11):
            a = np.zeros((48, 48, 48), np.uint8)
            b = np.zeros((48, 48, 48), np.uint8)
            idx = [slice(20, 23)] * 3
            a[tuple(idx)] = 1
            idx[axis] = slice(20 + 2 + gap, 23 + 2 + gap)
            b[tuple(idx)] = 1
            _check(a, b, 2, cuda)
    # random surfaces with D2 = 16: dense enough that everything is near
    vt = (rng.random((24, 20, 16)) < 0.5).astype(np.uint8)
    vp = (rng.random((24, 20, 16)) < 0.5).astype(np.uint8)
    _check(vt, vp, 2, cuda)
