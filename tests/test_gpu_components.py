"""GPU: connected-component counts (octm_components_u8, evaluate(components=...)) equal the oracle exactly."""
import numpy as np
import pytest

from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, synth
import components_oracle as co

pytestmark = pytest.mark.gpu

CONNS = (4, 8)


def _dev(a, cuda):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _counts(t, p, k, conn):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    out = suite.components(t, p, k, conn)
    torch.cuda.synchronize()
    assert out.connectivity == conn
    return out.n_comp.cpu().numpy().view(np.uint32), out.n_hit.cpu().numpy().view(np.uint32)


def _check(yt, yp, k, cuda, t=None, p=None, conns=CONNS, msg=""):
    t = _dev(yt, cuda) if t is None else t
    p = _dev(yp, cuda) if p is None else p
    got = {}
    for conn in conns:
        nc, nh = _counts(t, p, k, conn)
        ref_nc, ref_nh = co.label_counts(yt, yp, k, conn)
        np.testing.assert_array_equal(nc, ref_nc, err_msg=f"{msg} n_comp conn={conn}")
        np.testing.assert_array_equal(nh, ref_nh, err_msg=f"{msg} n_hit conn={conn}")
        got[conn] = nc
    return got


def test_random_masks(cuda):
    """1 x 1 to 20 x 20 and 1-row / 1-column strips: an absent class, a class filling the map, identical maps."""
    rng = np.random.default_rng(201)
    shapes = [(1, 1), (1, 37), (29, 1), (1, 600), (700, 1)] + [tuple(rng.integers(1, 21, size=2)) for _ in range(20)]
    for h, w in shapes:
        n = 6
        a = (rng.random((n, h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8)
        b = (rng.random((n, h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8)
        a[0] = 0
        b[1] = 1
        a[2] = b[2]
        a[3] = rng.integers(0, 4, size=(h, w))
        b[3] = rng.integers(0, 4, size=(h, w))
        _check(a, b, 4, cuda, msg=f"{h}x{w}")


def _serpentine(h, w):
    m = np.zeros((h, w), np.uint8)
    m[::2] = 1
    for y in range(1, h, 2):
        m[y, w - 1 if (y // 2) % 2 == 0 else 0] = 1
    return m


def test_adversarial_shapes(cuda):
    h, w = 496, 512
    serp = _serpentine(h, w)
    got = _check(serp[None], serp[None], 2, cuda, msg="serpentine")
    assert got[4][0, 1].tolist() == [1, 1]                           # one component over the whole map
    u = np.zeros((1, 40, 64), np.uint8)                                # U shapes joined only in the last row
    for x0 in range(2, 60, 8):
        u[0, :, x0] = u[0, :, x0 + 4] = 1
        u[0, 39, x0:x0 + 5] = 1
    inv = u[:, ::-1].copy()                                            # inverted: the arms split off
    got = _check(np.concatenate([u, inv]), np.concatenate([inv, u]), 2, cuda, msg="U")
    assert got[4][:, 1, 0].tolist() == [8, 8]
    diag = np.zeros((1, 48, 80), np.uint8)                             # diagonal-only chains
    for s in range(0, 80, 6):
        for y in range(48):
            if s + y < 80:
                diag[0, y, s + y] = 1
    got = _check(diag, np.roll(diag, 1, axis=2), 2, cuda, msg="diagonal")
    assert got[8][0, 1, 0] < got[4][0, 1, 0]
    for bh, bw in ((7, 9), (496, 512), (33, 1000)):
        yy, xx = np.mgrid[:bh, :bw]
        board = ((yy + xx) % 2).astype(np.uint8)[None]
        got = _check(board, 1 - board, 2, cuda, msg=f"board {bh}x{bw}")
        assert got[8][0].tolist() == [[1, 1], [1, 1]]
        assert got[4][0, :, 0].tolist() == [(bh * bw + 1) // 2, bh * bw // 2]
    stripes = (np.arange(512) % 2).astype(np.uint8)[None, None].repeat(64, axis=1)   # single-pixel vertical stripes
    got = _check(stripes, stripes[:, ::-1].copy(), 2, cuda, msg="stripes")
    assert got[4][0, :, 0].tolist() == [256, 256]


def test_labels_at_or_above_k_are_not_counted(cuda):
    rng = np.random.default_rng(205)
    yt = rng.integers(0, 3, size=(4, 50, 70)).astype(np.uint8)
    yp = rng.integers(0, 3, size=(4, 50, 70)).astype(np.uint8)
    yt[rng.random(yt.shape) < 0.1] = 255
    yp[rng.random(yp.shape) < 0.1] = 3
    _check(yt, yp, 3, cuda, msg="ignore labels")


def test_unaligned_and_odd_widths(cuda):
    rng = np.random.default_rng(206)
    for w in (50, 513, 1000, 1025):
        yt = rng.integers(0, 5, size=(4, 21, w)).astype(np.uint8)
        yp = yt.copy()
        yp[rng.random(yp.shape) < 0.2] = 2
        _check(yt, yp, 5, cuda, msg=f"W={w}")
    yt = rng.integers(0, 3, size=(3, 30, 512)).astype(np.uint8)
    yp = yt.copy()
    yp[rng.random(yp.shape) < 0.05] = 1
    pad = np.zeros(1, np.uint8)
    flat_t, flat_p = _dev(np.concatenate([pad, yt.ravel()]), cuda), _dev(np.concatenate([pad, yp.ravel()]), cuda)
    t, p = flat_t[1:].view(3, 30, 512), flat_p[1:].view(3, 30, 512)      # one byte off 16-byte alignment
    assert t.data_ptr() % 16 != 0 and p.data_ptr() % 16 != 0
    _check(yt, yp, 3, cuda, t, p, msg="unaligned")


@pytest.mark.parametrize("case", ["clean", "noise", "ragged", "lesion", "k10_w1000", "k16_w2048", "uniform"])
def test_workloads(cuda, case):
    import torch
    if case == "clean":
        t, p = synth.layered_pair_device(4, 496, 512, 8, seed=4004, device=cuda)
        yt, yp, k = t.cpu().numpy(), p.cpu().numpy(), 8
        got = _check(yt, yp, k, cuda, t, p, msg=case)
        present = np.stack([[np.isin(c, m) for c in range(k)] for m in yt])
        for conn in CONNS:                                       # a clean layer band is one region
            assert (got[conn][..., 0][present] == 1).all() and (got[conn][..., 0][~present] == 0).all()
        return
    if case == "noise":
        t, p = synth.layered_pair_device(3, 496, 512, 8, seed=4004, device=cuda, noise=0.002)
        yt, yp, k = t.cpu().numpy(), p.cpu().numpy(), 8
    elif case == "ragged":
        t, p = synth.ragged_pair_device(3, 496, 512, 8, seed=4005, device=cuda)
        yt, yp, k = t.cpu().numpy(), p.cpu().numpy(), 8
    elif case == "lesion":
        yt, yp = synth.lesion_pair(4, 496, 512, 4, seed=3003, single_blob_interior=False)
        k, t, p = 4, None, None
    elif case == "k10_w1000":
        yt, yp = synth.layered_pair(2, 128, 1000, 10, seed=214, noise=0.002)
        k, t, p = 10, None, None
    elif case == "k16_w2048":
        yt, yp = synth.layered_pair(2, 64, 2048, 16, seed=217, noise=0.005, min_gap=1)
        k, t, p = 16, None, None
    else:
        g = torch.Generator(device=cuda).manual_seed(4006)
        t, p = (torch.randint(0, 8, (2, 496, 512), generator=g, device=cuda, dtype=torch.uint8) for _ in range(2))
        yt, yp, k = t.cpu().numpy(), p.cpu().numpy(), 8
    _check(yt, yp, k, cuda, t, p, msg=case)


def test_suite_integration(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist, suite
    yt, yp = synth.lesion_pair(12, 64, 128, 4, seed=221, single_blob_interior=False)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    base = suite.evaluate(t, p, 4)
    assert base.component_connectivity is None and "component_f1" not in base.metrics()
    bm, bi = base.metrics(), base.integers()
    for conn in CONNS:
        res = suite.evaluate(t, p, 4, components=conn)
        assert res.component_connectivity == conn
        m, mh, ints = res.metrics(), res.metrics_host(), res.integers()
        assert set(m) - set(bm) == set(derive.COMPONENT_METRICS)
        for key in mh:
            np.testing.assert_array_equal(m[key], mh[key], err_msg=key)
        ref_nc, ref_nh = co.label_counts(yt, yp, 4, conn)
        np.testing.assert_array_equal(ints["component_count"], ref_nc)
        np.testing.assert_array_equal(ints["component_hits"], ref_nh)
        assert ints["component_count"].dtype == np.uint32 and ints["component_count"].shape == (12, 4, 2)
        for key, v in derive.component_metrics(ref_nc, ref_nh).items():
            assert m[key].shape == (12, 4)
            np.testing.assert_array_equal(m[key], v, err_msg=key)
        for key, v in bm.items():                    # everything else is what evaluate() gives without it
            np.testing.assert_array_equal(m[key], v, err_msg=key)
        assert set(ints) - set(bi) == {"component_count", "component_hits"}
        for key, v in bi.items():
            assert np.array_equal(ints[key].view(np.uint8), v.view(np.uint8)), key
        np.testing.assert_array_equal(res.totals_host(), base.totals_host())
        for contours, sd in ((False, None), ("all", 1.0)):          # independent of the other optional passes
            other = suite.evaluate(t, p, 4, contours=contours, surface_dice=sd, components=conn).integers()
            np.testing.assert_array_equal(other["component_count"], ref_nc)
            np.testing.assert_array_equal(other["component_hits"], ref_nh)
        host = suite.evaluate_host(yt, yp, 4, chunk_items=5, components=conn)
        assert host.component_connectivity == conn
        for key, v in m.items():
            np.testing.assert_array_equal(host.metrics()[key], v, err_msg=key)
        for key, v in ints.items():
            np.testing.assert_array_equal(host.integers()[key], v, err_msg=key)
        again = suite.evaluate(t, p, 4, components=conn).integers()      # two runs give equal counts
        np.testing.assert_array_equal(again["component_count"], ints["component_count"])
        np.testing.assert_array_equal(again["component_hits"], ints["component_hits"])
        tot = dist.component_totals(res, 1)
        np.testing.assert_array_equal(tot["component_count"], ref_nc.sum(0))
        np.testing.assert_array_equal(tot["component_hits"], ref_nh.sum(0))
    empty = suite.evaluate(t[:0], p[:0], 4, components=8)
    assert empty.metrics()["component_f1"].shape == (0, 4)
    for bad in (0, 6, "8", True):
        with pytest.raises(ValueError):
            suite.evaluate(t, p, 4, components=bad)
    torch.cuda.synchronize()


def test_kernel_launches(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, _lib
    yt, yp = synth.lesion_pair(4, 96, 128, 4, seed=231, single_blob_interior=False)
    t, p = _dev(yt, cuda), _dev(yp, cuda)
    lib = _lib.load()
    lib.octm_label_pass_seed_policy(2)          # the label pass's route must not depend on call history here
    try:
        with _lib.kernel_profile() as prof:
            suite.evaluate(t, p, 4).metrics()
            torch.cuda.synchronize()
        before = {name: c for name, (c, _) in prof.kernels.items()}
        assert "components_kernel" not in before
        with _lib.kernel_profile() as prof:
            suite.evaluate(t, p, 4, components=4).metrics()
            torch.cuda.synchronize()
        after = {name: c for name, (c, _) in prof.kernels.items()}
    finally:
        lib.octm_label_pass_seed_policy(0)
    assert after.pop("components_kernel") == 1
    assert after == before                                    # every other launch as without components
    with _lib.kernel_profile() as prof:
        suite.evaluate_host(yt, yp, 4, chunk_items=2, components=8).metrics()
        torch.cuda.synchronize()
    assert prof.kernels["components_kernel"][0] == 2           # one launch per chunk
