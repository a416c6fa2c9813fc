"""GPU parity: 3-D surface distances with a voxel spacing and the volumetric normalized surface Dice
(``suite.surface_distance_3d(spacing=..., tolerances=...)``) against ``tests/surface3d_spacing_oracle.py``.

At dyadic spacings every product and sum is exact, so counts, max, both order statistics of the 95th percentile,
``n_surf`` and ``n_within`` are bit-exact and the distance sums agree to 1e-12 relative.  At OCT-like spacings the
squared-distance statistics agree to 1e-12 relative (the oracle's nearest voxel is scipy's, chosen in scipy's rounding),
and the counts are exact on inputs where no distance lies within 1e-9 relative of a tolerance, which each such case
asserts.  Each case asserts on its inputs that it reaches the route it is named for (csrc/edt3d.cu, physical spacing:
pass 1 vectorised when D2 % 16 == 0 and the source volume is 16-byte aligned, byte-wise otherwise; passes 2 and 3 keep
stacks of MAX_LINE entries).
"""
import numpy as np
import pytest

import surface3d_spacing_oracle as sso
from retinal_oct_image_segmentation_via_deep_learning_b200 import synth

pytestmark = pytest.mark.gpu
RTOL = 1e-6
MAX_LINE = 2048         # kMaxLine in edt3d.cu
KEYS = ("sq_pred_to_true", "sq_true_to_pred")       # direction 0, direction 1
OCT = (0.0039, 0.0117, 0.047)                       # mm: axial, lateral, between B-scans


def _to(cuda, *vols):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(v)).to(cuda) for v in vols)


def _misaligned(t):
    import torch
    buf = torch.empty(t.numel() + 1, dtype=torch.uint8, device=t.device)
    v = buf[1:].view(t.shape).copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 2 == 1
    return v


def _same(got, want, exact):
    if exact:
        return got == want
    return abs(got - want) <= 1e-12 * abs(want)


def _check(vt, vp, k, spacing, taus, cuda, vols=None, exact=True):
    """Run on (vt, vp), or on device tensors ``vols`` with the same contents, and compare every output of every class
    and direction with the oracle.  Returns (outputs, {class: oracle result})."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    ints = suite.surface_distance_3d(*(vols if vols is not None else _to(cuda, vt, vp)), k, spacing=spacing,
                                     tolerances=taus)
    m = suite.surface_metrics_3d(ints)
    n_pts = ints["n_pts"].cpu().numpy().view(np.uint32)
    max_sq, p95, sums = (ints[key].cpu().numpy() for key in ("max_sq", "p95_sq", "sum_dist"))
    assert max_sq.dtype == p95.dtype == np.float64
    if taus:
        n_surf = ints["n_surf"].cpu().numpy()
        n_within = ints["n_within"].cpu().numpy()
        assert n_within.shape == (k, 2, len(taus))
    else:
        assert "n_surf" not in ints and "surface_dice" not in m
    refs = {}
    for c in range(k):
        ref = refs[c] = sso.class_metrics(vt, vp, c, spacing, taus or ())
        if taus:
            assert tuple(n_surf[c]) == tuple(ref["n_surf"]), (c, n_surf[c], ref["n_surf"])
            np.testing.assert_array_equal(m["surface_dice"][c], ref["surface_dice"], err_msg=f"surface_dice {c}")
        if ref["sq_pred_to_true"] is None or ref["sq_true_to_pred"] is None:
            assert not (n_pts[c].any() or max_sq[c].any() or p95[c].any() or sums[c].any()), c
            assert not taus or not n_within[c].any(), c
            assert np.isnan(m["hausdorff_distance"][c]) and np.isnan(m["assd"][c])
            continue
        for d, key in enumerate(KEYS):
            s = np.sort(ref[key])
            n = len(s)
            lo = int(np.floor((n - 1) * 0.95))
            assert n_pts[c, 1 - d] == n, (c, d)
            assert _same(max_sq[c, d], s[-1], exact), (c, d, max_sq[c, d], s[-1])
            for j, want in enumerate((s[lo], s[min(lo + 1, n - 1)])):
                assert _same(p95[c, d, j], want, exact), (c, d, j, p95[c, d, j], want)
            np.testing.assert_allclose(sums[c, d], np.sqrt(s).sum(), rtol=1e-12, err_msg=f"sum_dist {c} {d}")
            if taus and not exact:          # counts are exact where no distance is near a tolerance
                e = np.sqrt(s)
                for t in taus:
                    assert not np.any(np.abs(e - t) <= 1e-9 * t), (c, d, t)
        if taus:
            assert np.array_equal(n_within[c], ref["n_within"]), (c, n_within[c], ref["n_within"])
        assert _same(m["hausdorff_distance"][c], ref["hausdorff_distance"], exact), c
        for name in ("hausdorff_distance_95", "assd"):
            np.testing.assert_allclose(m[name][c], ref[name], rtol=RTOL, atol=0, err_msg=f"{name} class {c}")
    return ints, refs


def _lesion_volume(shape, k, seed):
    """Fluid-like ellipsoid blobs of classes 1..k-1 on background 0; the prediction's blobs are shifted and resized."""
    rng = np.random.default_rng(seed)
    grid = np.indices(shape, dtype=np.float64)
    vt = np.zeros(shape, np.uint8)
    vp = np.zeros(shape, np.uint8)
    for c in range(1, k):
        for _ in range(2):
            ctr = rng.uniform(0.2, 0.8, 3) * shape
            rad = rng.uniform(0.08, 0.25, 3) * shape
            r2 = sum(((grid[i] - ctr[i]) / rad[i]) ** 2 for i in range(3))
            vt[r2 <= 1] = c
            ctr2 = ctr + rng.normal(0, 1.5, 3)
            rad2 = rad * rng.uniform(0.8, 1.2, 3)
            r2 = sum(((grid[i] - ctr2[i]) / rad2[i]) ** 2 for i in range(3))
            vp[r2 <= 1] = c
    return vt, vp


def _tie_tolerance(vt, vp, cls, spacing):
    """A tolerance equal to a distance that occurs in direction 0 of class ``cls`` (the median one)."""
    d = np.sort(sso.squared_distances(vp == cls, vt == cls, spacing))
    return float(np.sqrt(d[len(d) // 2]))


@pytest.mark.parametrize("spacing", [(0.5, 1.0, 2.0), (1.0, 1.0, 4.0)])
def test_dyadic_spacings(cuda, spacing):
    for vt, vp in (synth.layered_volume_pair(40, 36, 32, 5, seed=81), _lesion_volume((36, 40, 24), 4, seed=82)):
        tie = _tie_tolerance(vt, vp, 1, spacing)
        taus = (0.0, tie, 1.5, 6.0)
        _, refs = _check(vt, vp, int(max(vt.max(), vp.max())) + 1, spacing, taus, cuda)
        assert np.any(np.sqrt(refs[1]["sq_pred_to_true"]) == tie)     # '<=' is exercised at the tie


def test_oct_like_spacing(cuda):
    for vt, vp in (synth.layered_volume_pair(48, 40, 32, 5, seed=83), _lesion_volume((40, 36, 20), 3, seed=84)):
        k = int(max(vt.max(), vp.max())) + 1
        _, refs = _check(vt, vp, k, OCT, (0.01, 0.02, 0.05), cuda, exact=False)
        _check(vt, vp, k, OCT, None, cuda, exact=False)
        within = np.array([refs[c]["n_within"] for c in range(k)])
        assert within.any() and (within < np.array([refs[c]["n_surf"][::-1, None] for c in range(k)])).any()


def test_anisotropy_changes_the_nearest_voxel(cuda):
    """30:1 along D2: the y_true voxel one step along D2 is nearest in index space, the one five steps along D0 in
    physical space."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    vt = np.zeros((24, 12, 16), np.uint8)
    vp = np.zeros((24, 12, 16), np.uint8)
    vp[10, 5, 5] = 1
    vt[10, 5, 6] = 1                                   # one step along D2
    vt[15, 5, 5] = 1                                   # five steps along D0
    ints, refs = _check(vt, vp, 2, (1.0, 1.0, 30.0), (5.0,), cuda)
    assert refs[1]["sq_pred_to_true"].tolist() == [25.0]
    assert float(ints["max_sq"][1, 0]) == 25.0
    unit = suite.surface_distance_3d(*_to(cuda, vt, vp), 2, spacing=(1, 1, 1))
    assert float(unit["max_sq"][1, 0]) == 1.0                          # the unit-spacing answer differs


def test_unit_spacing_is_the_integer_path(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    rng = np.random.default_rng(85)
    vols = [synth.layered_volume_pair(40, 24, 32, 4, seed=86),
            ((rng.random((20, 33, 17)) < 0.3).astype(np.uint8) * 3, (rng.random((20, 33, 17)) < 0.3).astype(np.uint8) * 3)]
    vt = np.zeros((120, 80, 12), np.uint8)             # far apart: the integer path's global histogram bins
    vp = np.zeros((120, 80, 12), np.uint8)
    vt[0:6, 0:5, :] = 1
    vp[100:120, 70:80, 3:9] = 1
    vols.append((vt, vp))
    for vt, vp in vols:
        t, p = _to(cuda, vt, vp)
        ref = suite.surface_distance_3d(t, p, 4)
        for kw in ({"spacing": (1, 1, 1)}, {"tolerances": (1.0, 2.5)}):
            got = suite.surface_distance_3d(t, p, 4, **kw)
            assert torch.equal(got["n_pts"], ref["n_pts"])
            for key in ("max_sq", "p95_sq"):
                assert torch.equal(got[key], ref[key].to(torch.int64).to(torch.float64)), key
            torch.testing.assert_close(got["sum_dist"], ref["sum_dist"], rtol=1e-12, atol=0)
    assert ref["max_sq"].max() >= 8192


def test_long_lines(cuda):
    """Lines of MAX_LINE voxels along D0 (pass-3 stacks) and D1 (pass-2 stacks): a whole line of class 2 in one corner
    of y_true and in the opposite one of y_pred, every voxel of it surface and equally far from the other, so every
    envelope over such lines keeps every site; class 1 sparse random."""
    rng = np.random.default_rng(87)
    for shape in ((MAX_LINE, 3, 16), (3, MAX_LINE, 16)):
        axis = int(np.argmax(shape))
        vt = (rng.random(shape) < 0.001).astype(np.uint8)
        vp = (rng.random(shape) < 0.001).astype(np.uint8)
        lt, lp = [0, 0, 0], [-1, -1, -1]
        lt[axis] = lp[axis] = slice(None)
        vt[tuple(lt)] = 2
        vp[tuple(lp)] = 2
        spacing = (0.5, 2.0, 0.25)
        _, refs = _check(vt, vp, 3, spacing, (1.0, 4.0), cuda)
        w = sso.weights(spacing)
        across = sum(w[i] * (s - 1) ** 2 for i, s in enumerate(shape) if i != axis)
        for key in KEYS:
            assert refs[2][key].tolist() == [across] * MAX_LINE, key


def test_misaligned_volumes(cuda):
    """Byte-wise pass 1 (D2 % 16 != 0, or volumes at odd addresses) against the vectorised one: identical outputs."""
    import torch
    vt, vp = synth.layered_volume_pair(40, 24, 32, 4, seed=88)
    t, p = _to(cuda, vt, vp)
    assert t.data_ptr() % 16 == 0 and p.data_ptr() % 16 == 0
    ref, _ = _check(vt, vp, 4, (0.5, 1.0, 2.0), (1.0, 3.0), cuda, vols=(t, p))
    for vols in ((t, _misaligned(p)), (_misaligned(t), _misaligned(p))):
        got, _ = _check(vt, vp, 4, (0.5, 1.0, 2.0), (1.0, 3.0), cuda, vols=vols)
        for key in ref:
            assert torch.equal(got[key], ref[key]), key
    vt, vp = synth.layered_volume_pair(30, 20, 21, 4, seed=89)          # D2 % 16 != 0
    _check(vt, vp, 4, OCT, (0.01, 0.03), cuda, exact=False)


def test_empty_surfaces(cuda):
    """Class 1 only in y_true: no distances (n_pts 0, NaN metrics), NSD 0 with the true n_surf; class 2 in neither:
    NSD NaN; class 3 in y_pred only."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    vt = np.zeros((20, 18, 16), np.uint8)
    vp = np.zeros((20, 18, 16), np.uint8)
    vt[3:9, 4:10, 2:7] = 1
    vp[10:15, 2:6, 8:14] = 3
    vt[15:18, 12:16, 9:12] = 4
    vp[14:18, 12:16, 9:13] = 4
    ints, refs = _check(vt, vp, 5, (0.5, 1.0, 2.0), (1.0, 2.0), cuda)
    m = suite.surface_metrics_3d(ints)
    ns = ints["n_surf"].cpu().numpy()
    assert ns[1, 0] == refs[1]["n_surf"][0] > 0 and ns[1, 1] == 0 and ns[3, 0] == 0 and ns[3, 1] > 0
    assert not ints["n_pts"][1].any() and not ints["n_pts"][3].any()
    assert (m["surface_dice"][1] == 0).all() and (m["surface_dice"][3] == 0).all()
    assert np.isnan(m["surface_dice"][2]).all() and not ns[2].any()
    assert np.isnan(m["hausdorff_distance"][1]) and np.isnan(m["hausdorff_distance_95"][3])
    assert np.isfinite(m["hausdorff_distance"][4]) and (m["surface_dice"][4] > 0).all()


def test_class_255_and_bool_inputs(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    vt = np.zeros((24, 16, 32), np.uint8)
    vp = np.zeros((24, 16, 32), np.uint8)
    vt[4:12, 2:8, 20:32] = 255                         # touches the last D2 face (the vectorised pass 1's padding)
    vp[5:12, 2:9, 18:31] = 255
    vp[20, 14, 1] = 255
    vt[14:20, 9:14, 3:9] = 127
    vp[14:21, 9:14, 4:9] = 127
    _check(vt, vp, 256, (0.5, 1.0, 2.0), (1.0,), cuda)
    t, p = _to(cuda, vt == 255, vp == 255)
    assert t.dtype == torch.bool
    as_bool = suite.surface_distance_3d(t, p, 2, spacing=OCT, tolerances=(0.01,))
    as_u8 = suite.surface_distance_3d(t.to(torch.uint8), p.to(torch.uint8), 2, spacing=OCT, tolerances=(0.01,))
    for key in as_u8:
        assert torch.equal(as_bool[key], as_u8[key]), key
    _check((vt == 255).astype(np.uint8), (vp == 255).astype(np.uint8), 2, OCT, (0.01,), cuda, vols=(t, p), exact=False)


def test_unit_ranges_add_up_and_repeat(cuda):
    """Disjoint unit ranges add up to the full call; each single unit writes its own entries only; two calls are
    bit-identical (sums, order statistics and counts included)."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    vt, vp = _lesion_volume((32, 28, 24), 4, seed=90)
    t, p = _to(cuda, vt, vp)
    kw = {"spacing": OCT, "tolerances": (0.01, 0.02, 0.04)}
    full = suite.surface_distance_3d(t, p, 4, **kw)
    a = suite.surface_distance_3d(t, p, 4, units=(0, 3), **kw)
    b = suite.surface_distance_3d(t, p, 4, units=(3, 8), **kw)
    for key in full:
        assert torch.equal(a[key] + b[key], full[key]), key
    for u in range(8):
        c, d = divmod(u, 2)
        one = suite.surface_distance_3d(t, p, 4, units=(u, u + 1), **kw)
        for key, at in (("n_pts", (c, 1 - d)), ("n_surf", (c, 1 - d)), ("max_sq", (c, d)), ("p95_sq", (c, d)),
                        ("sum_dist", (c, d)), ("n_within", (c, d))):
            mine = torch.zeros(full[key].shape, dtype=torch.bool, device=cuda)
            mine[at] = True
            assert torch.equal(one[key][mine], full[key][mine]), (u, key)
            assert not one[key][~mine].any(), (u, key)
    for _ in range(2):
        again = suite.surface_distance_3d(t, p, 4, **kw)
        for key in full:
            assert torch.equal(again[key], full[key]), key
