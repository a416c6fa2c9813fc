"""CPU tier of the per-sector layer thickness: argument checks of ``octm_sector_thickness_i32`` (OCTM_ERR_INVALID before
any CUDA call), the ETDRS region map against a per-A-scan loop, the host epilogue and summary against plain numpy, the
Python argument checks, the oracle against a pure-Python loop, and the two-rank packing of
``dist.sector_thickness_totals`` over gloo."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest

import sector_thickness_oracle as sto
from oracle import labelmap_oracle as lo


@pytest.fixture(scope="module")
def lib():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails
DUKE = (61, 768, (0.1185, 0.00387, 0.00772))       # B-scans, width, (sb, sy, sx) in mm
HCMS = (49, 1024, (0.1229, 0.00387, 0.00583))


def _err(lib):
    return lib.octm_last_error().decode()


# ------------------------------------------------------------------------------------------ C ABI
def _call(lib, n=0, k=8, h=496, w=768, ipv=1, nr=9, groups=((0, 0), (1, 7)), ng=None, null=()):
    """``n`` = 0 by default: a call that passes every check returns OCTM_OK before any CUDA call."""
    p = {name: None if name in null else FAKE for name in ("bnd_true", "bnd_pred", "region", "sums")}
    flat = [c for pair in groups for c in pair]
    grp = None if "groups" in null else (ctypes.c_int32 * max(1, len(flat)))(*flat)
    return lib.octm_sector_thickness_i32(p["bnd_true"], p["bnd_pred"], n, k, h, w, ipv, p["region"], nr, grp,
                                         len(groups) if ng is None else ng, p["sums"], None, None)


def test_abi_checks(lib):
    assert _call(lib) == 0
    assert _call(lib, n=0, ipv=61) == 0
    for kw in ({"n": -1}, {"h": 0}, {"w": 0}):
        assert _call(lib, **kw) == -1 and "shape" in _err(lib), kw
    for k in (1, 17):
        assert _call(lib, k=k, groups=((0, 0),)) == -1 and "num_classes" in _err(lib), k
    assert _call(lib, n=10, ipv=3) == -1 and "items_per_volume" in _err(lib)
    assert _call(lib, ipv=0) == -1 and "items_per_volume" in _err(lib)
    for nr in (0, 17):
        assert _call(lib, nr=nr) == -1 and "n_regions" in _err(lib), nr
    assert _call(lib, nr=16) == 0
    assert _call(lib, groups=()) == -1 and "n_groups" in _err(lib)
    assert _call(lib, groups=((0, 0),) * 17) == -1 and "n_groups" in _err(lib)
    assert _call(lib, groups=((0, 0),) * 16) == 0
    for bad in ((-1, 0), (3, 2), (0, 8), (8, 8)):
        assert _call(lib, groups=((0, 0), bad)) == -1 and "groups[1]" in _err(lib), bad
    assert _call(lib, groups=((7, 7), (0, 7))) == 0
    assert _call(lib, null=("groups",)) == -1 and "null" in _err(lib)
    # items_per_volume * W * H^2 < 2^53: 2^27 * 1 * 2^26 = 2^53 fails, one item less passes
    assert _call(lib, h=1 << 13, w=1, ipv=1 << 27) == -1 and "2^53" in _err(lib)
    assert _call(lib, h=1 << 13, w=1, ipv=(1 << 27) - 1) == 0
    assert _call(lib, h=3000, w=1024, ipv=1 << 20) == -1 and "2^53" in _err(lib)
    for name in ("bnd_true", "bnd_pred", "region", "sums"):
        assert _call(lib, n=1, null=(name,)) == -1 and "null" in _err(lib), name
        assert _call(lib, null=(name,)) == 0, name                     # an empty batch touches nothing


# ------------------------------------------------------------------------------------------ ETDRS grid
def _brute_regions(nb, w, spacing, center, radii):
    sb, _, sx = spacing
    cb, cx = center
    r0, r1, r2 = radii
    out = np.zeros((nb, w), np.uint8)
    for b in range(nb):
        for x in range(w):
            pb = (b - cb) * sb
            px = (x - cx) * sx
            d = pb * pb + px * px
            if abs(pb) > abs(px):
                q = 0 if pb < 0 else 2
            else:
                q = 1 if px > 0 else 3
            if d <= r0 * r0:
                out[b, x] = 0
            elif d <= r1 * r1:
                out[b, x] = 1 + q
            elif d <= r2 * r2:
                out[b, x] = 5 + q
            else:
                out[b, x] = 255
    return out


@pytest.mark.parametrize("geometry", [DUKE, HCMS], ids=["duke", "hcms"])
def test_regions_against_brute_force(geometry):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    nb, w, sp = geometry
    centers = [((nb - 1) / 2, (w - 1) / 2), (nb / 3, w * 0.6 + 0.25), (2.0, 40.5), (-5.0, w + 100.0), (nb - 1, 0)]
    for c in centers:
        got = derive.etdrs_regions(nb, w, sp, c)
        assert got.dtype == np.uint8 and got.shape == (nb, w)
        assert np.array_equal(got, _brute_regions(nb, w, sp, c, derive.ETDRS_RADII)), c
    # the centred grid covers every sector, and the 6 mm disc leaves the corners out
    full = derive.etdrs_regions(nb, w, sp, centers[0])
    assert set(np.unique(full).tolist()) == set(range(9)) | {255}
    # a centre far outside the scan leaves no A-scan in any region
    assert np.all(derive.etdrs_regions(nb, w, sp, (-1000.0, -1000.0)) == 255)


def test_radius_on_an_ascan_and_diagonal_ties():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    sp = (0.5, 0.004, 0.5)                      # dyadic: every position and r2 below is exact
    reg = derive.etdrs_regions(9, 9, sp, (4, 4), (1.0, 1.5, 2.0))
    assert reg[4, 4] == 0
    assert reg[4, 6] == 0 and reg[2, 4] == 0     # r2 = 1.0 == R0^2: on the circle is inside
    assert reg[4, 7] == 2 and reg[4, 1] == 4     # inner x+, x-
    assert reg[1, 4] == 1 and reg[7, 4] == 3     # inner b-, b+
    assert reg[4, 8] == 6 and reg[0, 4] == 5     # r2 = 4.0 == R2^2: the outer ring's edge is inside
    # |pb| == |px| goes to the x side
    assert reg[3, 5] == 0                        # r2 = 0.5 <= 1
    assert reg[2, 6] == 2 and reg[6, 6] == 2     # r2 = 2.0 <= 2.25: inner x+, from the b- and the b+ side
    assert reg[2, 2] == 4 and reg[6, 2] == 4     # inner x-
    assert reg[3, 7] == 6 and reg[5, 1] == 8     # r2 = 2.5: outer x+, x-
    assert reg[0, 0] == 255 and reg[8, 8] == 255


def test_sector_names_and_order():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    assert len(derive.ETDRS_SECTORS) == 9 and derive.ETDRS_SECTORS[0] == "center"
    assert derive.ETDRS_SECTORS[1:5] == ("inner_b-", "inner_x+", "inner_b+", "inner_x-")
    assert derive.ETDRS_SECTORS[5:] == ("outer_b-", "outer_x+", "outer_b+", "outer_x-")


# ------------------------------------------------------------------------------------------ epilogue and summary
def _random_sums(rng, v, g, r=9):
    n = rng.integers(0, 50, size=(v, g, r))
    n[0, :, 3] = 0                                           # an empty region in volume 0
    n[:, :, 8] = 0                                           # a region no volume covers
    t = rng.integers(0, 80, size=(v, g, r, 60))
    p = rng.integers(0, 80, size=(v, g, r, 60))
    mask = np.arange(60)[None, None, None, :] < n[..., None]
    d = (t - p) * mask
    return np.stack([n, (t * mask).sum(-1), (p * mask).sum(-1), np.abs(d).sum(-1), (d * d).sum(-1)], axis=-1)


def test_sector_thickness_epilogue_against_numpy():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    rng = np.random.default_rng(5)
    sums = _random_sums(rng, 4, 3)
    sp = (0.12, 0.0039, 0.0117)
    got = derive.sector_thickness(sums, sp)
    for v in range(4):
        for g in range(3):
            for r in range(9):
                n, st, spd, sa, ss = (int(x) for x in sums[v, g, r])
                if n == 0:
                    for key in ("thickness_true", "thickness_pred", "thickness_bias", "thickness_mae", "thickness_rmse",
                                "volume_true", "volume_pred"):
                        assert math.isnan(got[key][v, g, r]), key
                    continue
                assert got["thickness_true"][v, g, r] == st / n * sp[1]
                assert got["thickness_pred"][v, g, r] == spd / n * sp[1]
                assert got["thickness_bias"][v, g, r] == (spd - st) / n * sp[1]
                assert got["thickness_mae"][v, g, r] == sa / n * sp[1]
                assert got["thickness_rmse"][v, g, r] == math.sqrt(ss / n) * sp[1]
                assert got["volume_true"][v, g, r] == st * ((sp[0] * sp[1]) * sp[2])
                assert got["volume_pred"][v, g, r] == spd * ((sp[0] * sp[1]) * sp[2])
    assert np.array_equal(got["n_ascans"], sums[..., 0]) and got["n_ascans"].dtype == np.int64


def test_summary_against_numpy():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    rng = np.random.default_rng(6)
    per = derive.sector_thickness(_random_sums(rng, 5, 2), (0.12, 0.0039, 0.0117))
    summ = derive.sector_thickness_summary(per)
    cov = per["n_ascans"] > 0
    assert np.array_equal(summ["n_volumes"], cov.sum(0))
    assert np.all(np.isnan(summ["bias"][:, 8])) and np.all(summ["n_volumes"][:, 8] == 0)
    for name, src in (("abs_bias", np.abs(per["thickness_bias"])), ("bias", per["thickness_bias"]),
                      ("mae", per["thickness_mae"]), ("rmse", per["thickness_rmse"]),
                      ("thickness_true", per["thickness_true"]), ("thickness_pred", per["thickness_pred"])):
        for g in range(2):
            for r in range(8):
                vals = [src[v, g, r] for v in range(5) if cov[v, g, r]]
                acc = 0.0
                for x in vals:
                    acc += x
                assert summ[name][g, r] == acc / len(vals), (name, g, r)
    assert list(summ) == list(derive.SECTOR_SUMMARY) + ["n_volumes"]


# ------------------------------------------------------------------------------------------ Python argument checks
def test_python_argument_checks():
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, suite
    assert derive.spacing_3d([1, 2, 3]) == (1.0, 2.0, 3.0)
    for sp in ((1, 1), (1, 1, 1, 1), (0, 1, 1), (1, -1, 1), (1, 1, np.nan), (np.inf, 1, 1), "abc", None):
        with pytest.raises(ValueError, match="spacing"):
            derive.spacing_3d(sp)
    assert derive.etdrs_radii((0.5, 1.5, 3)) == (0.5, 1.5, 3.0)
    assert derive.etdrs_radii((1, 1, 1)) == (1.0, 1.0, 1.0)
    for r in ((0, 1, 2), (1, 0.5, 2), (1, 2, 1.5), (1, 2), (1, 2, np.inf), (-1, 1, 2), ("a", 1, 2)):
        with pytest.raises(ValueError, match="radii"):
            derive.etdrs_radii(r)
    assert derive.sector_groups(None, 3) == ((0, 0), (1, 1), (2, 2))
    assert derive.sector_groups([2, (1, 7), np.int64(0), [3, 3]], 8) == ((2, 2), (1, 7), (0, 0), (3, 3))
    for classes in ([], list(range(17)), [8], [-1], [(2, 1)], [(0, 1, 2)], [1.5], [(0, 8)], [True], ["a"]):
        with pytest.raises(ValueError, match="classes"):
            derive.sector_groups(classes, 8)
    assert derive.sector_centers(None, 2, 61, 768).tolist() == [[30.0, 383.5], [30.0, 383.5]]
    assert derive.sector_centers((1, 2.5), 3, 5, 5).tolist() == [[1.0, 2.5]] * 3
    assert derive.sector_centers([[1, 2], [3, 4]], 2, 5, 5).tolist() == [[1.0, 2.0], [3.0, 4.0]]
    for c in ((1, 2, 3), [[1, 2]], [[1, 2], [3, 4], [5, 6]], (np.nan, 1), "ab"):
        with pytest.raises(ValueError, match="center"):
            derive.sector_centers(c, 2, 5, 5)
    y = torch.zeros((2, 3, 4, 5), dtype=torch.uint8)
    with pytest.raises(ValueError, match="spacing"):
        suite.sector_thickness(y, y, 3, (1, 1))
    with pytest.raises(ValueError, match="radii"):
        suite.sector_thickness(y, y, 3, (1, 1, 1), radii=(3, 2, 1))
    with pytest.raises(ValueError, match="classes"):
        suite.sector_thickness(y, y, 3, (1, 1, 1), classes=[(0, 3)])
    with pytest.raises(TypeError, match="CUDA"):
        suite.sector_thickness(y, y, 3, (1, 1, 1))


# ------------------------------------------------------------------------------------------ oracle
def test_oracle_against_python_loop():
    rng = np.random.default_rng(11)
    v, b, h, w, k = 2, 3, 7, 6, 4
    yt = rng.integers(0, k, size=(v, b, h, w), dtype=np.uint8)
    yp = rng.integers(0, k, size=(v, b, h, w), dtype=np.uint8)
    regions = rng.integers(0, 5, size=(v, b, w), dtype=np.uint8)
    regions[0, 0, :2] = 255
    groups = ((0, 0), (1, 2), (0, 3), (3, 3))
    sums, maps = sto.sector_sums(yt, yp, k, groups, regions, 4)       # code 4 counts nowhere
    assert np.array_equal(sums, sto.python_sums(yt, yp, groups, regions, 4))
    for i in range(v):
        for j in range(b):
            ct = lo.column_thickness(yt[i, j], k)
            assert np.array_equal(maps[i, j, 0, 1], ct[1] + ct[2])
            assert np.array_equal(maps[i, j, 0, 2], np.full(w, h))
            # the thickness of classes f..l is b_{l+1} - b_f of the boundary rows
            bt = np.concatenate([[np.zeros(w, np.int64)], lo.boundaries(yt[i, j], k), [np.full(w, h)]])
            for gi, (f, last) in enumerate(groups):
                assert np.array_equal(maps[i, j, 0, gi], bt[last + 1] - bt[f])


# ------------------------------------------------------------------------------------------ several ranks (gloo)
V, B, H, W, K = 5, 3, 12, 10, 4
GROUPS = ((0, 0), (1, 2), (3, 3))
SPACING = (0.25, 0.004, 0.5)


def _volumes():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import synth
    yt, yp = synth.layered_pair(V * B, H, W, K, seed=21, noise=0.05)
    return yt.reshape(V, B, H, W), yp.reshape(V, B, H, W)


def _regions():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    return np.stack([derive.etdrs_regions(B, W, SPACING, (1 + 0.3 * v, 4.5 - v), (0.6, 1.2, 2.0)) for v in range(V)])


def _fake_out(s, e, bad):
    """What a rank's ``suite.sector_thickness`` result holds for volumes [s, e), built from the oracle on CPU tensors."""
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    yt, yp = _volumes()
    sums, _ = sto.sector_sums(yt[s:e], yp[s:e], K, GROUPS, _regions()[s:e], 9)
    cm = np.zeros((0, K, K), np.int64)
    if e > s:
        cm = np.stack([lo.confusion_matrix(yt[i, j], yp[i, j], K) for i in range(s, e) for j in range(B)]).astype(np.int64)
    if bad and len(cm):
        cm[0, 0, 0] -= 1                 # a pixel the label pass dropped
    return suite.SectorThicknessOut(torch.from_numpy(sums), None, GROUPS, SPACING, K, torch.from_numpy(cm), H * W)


def _worker(rank, world, port, q, bad_rank, n_vol, shift_rank):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
    s, e = odist.shard_range(n_vol, rank, world)
    first = s + (n_vol if rank == shift_rank else 0)          # a volume range outside [0, n_vol) on that rank
    try:
        res = odist.sector_thickness_totals(_fake_out(s, e, rank == bad_rank), world, first, n_vol)
        q.put((rank, "ok", res))
    except ValueError as err:
        q.put((rank, "ValueError", str(err)))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def _run(bad_rank, n_vol=V, shift_rank=-1):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, bad_rank, n_vol, shift_rank)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict((g[0], g[1:]) for g in (q.get(timeout=120) for _ in range(2)))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return got


def test_two_rank_packing_equals_one_process():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    got = _run(bad_rank=-1)
    one = odist.sector_thickness_totals(_fake_out(0, V, False), 1, 0, V)
    yt, yp = _volumes()
    want, _ = sto.sector_sums(yt, yp, K, GROUPS, _regions(), 9)
    assert np.array_equal(one["sums"], want)
    assert np.array_equal(one["summary"]["n_volumes"], (want[..., 0] > 0).sum(0))
    for r in range(2):
        status, res = got[r]
        assert status == "ok"
        assert np.array_equal(res["sums"], want)
        for part in ("metrics", "summary"):
            for key in one[part]:
                assert np.array_equal(res[part][key], one[part][key], equal_nan=True), (part, key)
        assert res["groups"] == GROUPS and res["spacing"] == SPACING
    assert np.array_equal(one["metrics"]["thickness_mae"], derive.sector_thickness(want, SPACING)["thickness_mae"],
                          equal_nan=True)


def test_invalid_label_on_one_rank_raises_on_every_rank():
    got = _run(bad_rank=1)
    assert [got[r][0] for r in range(2)] == ["ValueError", "ValueError"]
    assert all("label >= num_classes" in got[r][1] for r in range(2))


def test_rank_without_volumes():
    """One volume over two ranks: rank 1 holds none, joins the collective and returns the single-process result."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    empty = _fake_out(1, 1, False)
    assert tuple(empty.sums.shape) == (0, len(GROUPS), 9, 5) and empty.bad_label_items() == 0
    assert empty.integers()["sums"].shape == (0, len(GROUPS), 9, 5)
    got = _run(bad_rank=-1, n_vol=1)
    one = odist.sector_thickness_totals(_fake_out(0, 1, False), 1, 0, 1)
    for r in range(2):
        status, res = got[r]
        assert status == "ok"
        assert np.array_equal(res["sums"], one["sums"]) and res["sums"].shape == (1, len(GROUPS), 9, 5)
        for part in ("metrics", "summary"):
            for key in one[part]:
                assert np.array_equal(res[part][key], one[part][key], equal_nan=True), (part, key)


def test_bad_volume_range_on_one_rank_raises_on_every_rank():
    got = _run(bad_rank=-1, shift_rank=0)
    assert [got[r][0] for r in range(2)] == ["ValueError", "ValueError"]
    assert all("outside [0, 5)" in got[r][1] for r in range(2))
