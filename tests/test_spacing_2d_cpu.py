"""CPU tier of the B-scan pixel spacing: argument checks in Python and in the C ABI (OCTM_ERR_INVALID before any CUDA
call), the spacing oracle against a pure-Python search, the host epilogue with a spacing, MetaImage spacing of
``evaluate_files`` and the dataset-level scaling of ``dist.unpack`` over gloo."""
import ctypes
import os
import socket

import numpy as np
import pytest

import spacing_2d_oracle as so
from oracle.contours_oracle import directed_sq_distances


@pytest.fixture(scope="module")
def lib():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails
OCT = (0.0039, 0.0117)           # mm: axial (rows), lateral (columns)


def _err(lib):
    return lib.octm_last_error().decode()


# ------------------------------------------------------------------------------------------ C ABI
def _distance(lib, n=0, k=2, max_pts=64, h=16, w=16, spacing=(1.0, 1.0), null=()):
    """``n`` = 0 by default: a call that passes every check returns OCTM_OK before any CUDA call."""
    p = {name: None if name in null else FAKE for name in ("verts", "n_pts", "max_sq", "p95_sq", "sum_dist", "d2")}
    sp = None if "spacing" in null else (ctypes.c_double * 2)(*spacing)
    return lib.octm_contour2d_distance_spacing(p["verts"], p["n_pts"], n, k, max_pts, h, w, sp, p["max_sq"], p["p95_sq"],
                                               p["sum_dist"], p["d2"], 0, None)


def test_distance_abi_checks(lib):
    assert _distance(lib) == 0
    assert _distance(lib, spacing=OCT) == 0
    for kw in ({"n": -1}, {"k": 0}, {"max_pts": 7}):
        assert _distance(lib, **kw) == -1 and "shape" in _err(lib), kw
    for kw in ({"h": 0}, {"w": 8193}):
        assert _distance(lib, **kw) == -1 and "8192" in _err(lib), kw
    for sp in ((0.0, 1.0), (1.0, -0.5), (float("nan"), 1.0), (1.0, float("inf")), (-0.0, 1.0)):
        assert _distance(lib, spacing=sp) == -1 and "finite and > 0" in _err(lib), sp
    for sp in ((1e-300, 1.0), (1.0, 1e300), (5e-324, 1.0), (1e-155, 1.0)):
        assert _distance(lib, spacing=sp) == -1 and "square" in _err(lib), sp
    assert _distance(lib, spacing=(1e153, 1.0), h=8192, w=16) == -1 and "diagonal" in _err(lib)
    assert _distance(lib, spacing=(1e150, 1e-150)) == 0
    assert _distance(lib, null=("spacing",)) == -1 and "null" in _err(lib)
    for name in ("verts", "n_pts", "max_sq", "p95_sq", "sum_dist", "d2"):
        assert _distance(lib, n=1, null=(name,)) == -1, name
        assert "null" in _err(lib) or "required" in _err(lib), name
        assert _distance(lib, null=(name,)) == 0, name                 # an empty batch touches nothing


def _surface(lib, n=0, spacing=(1.0, 1.0), taus=(1.0,), ntau=None, null=()):
    sp = None if "spacing" in null else (ctypes.c_double * 2)(*spacing)
    tol = None if "tolerances" in null else (ctypes.c_double * max(1, len(taus)))(*taus)
    return lib.octm_surface_dice_spacing_u8(FAKE, FAKE, n, 16, 16, 3, sp, tol, len(taus) if ntau is None else ntau,
                                            FAKE, FAKE, None)


def test_surface_dice_abi_checks(lib):
    assert _surface(lib) == 0
    for name in ("spacing", "tolerances"):
        assert _surface(lib, null=(name,)) == -1 and "null" in _err(lib), name
    for sp in ((0.0, 1.0), (1.0, float("nan")), (1e-300, 1.0)):
        assert _surface(lib, spacing=sp) == -1 and "spacing" in _err(lib), sp
    assert _surface(lib, taus=(1, 2, 3, 4, 5)) == -1 and "n_tolerances" in _err(lib)
    assert _surface(lib, taus=(1.0,), ntau=0) == -1 and "n_tolerances" in _err(lib)
    for taus in ((float("nan"),), (-0.5,), (float("inf"),)):
        assert _surface(lib, taus=taus) == -1 and "tolerances[0]" in _err(lib), taus
    # (1, 1): 16 lattice offsets reach tau < 8.5; 8 and the largest double below 8.5 are fine
    assert _surface(lib, taus=(8.0, np.nextafter(8.5, 0))) == 0
    assert _surface(lib, taus=(0.0, 8.5)) == -1 and "tolerances[1]" in _err(lib)
    assert "largest tolerance allowed is 8.4999999999999982" in _err(lib)
    # OCT spacing: the rows (3.9 um) bound the reach at sqrt(0.0039**2 * 289 / 4) = 0.03315 mm
    lim = float(np.nextafter(np.sqrt(OCT[0] * OCT[0] * 289 / 4.0), 0))
    assert _surface(lib, spacing=OCT, taus=(lim,)) == 0
    assert _surface(lib, spacing=OCT, taus=(np.nextafter(lim, 1),)) == -1 and "largest tolerance" in _err(lib)


def test_derive_abi_checks(lib):
    def call(sp):
        arr = None if sp is None else (ctypes.c_double * 2)(*sp)
        return lib.octm_derive_metrics_spacing(FAKE, None, None, None, None, None, None, None, None, 0, 8, 8, 3, arr,
                                               FAKE, None, None, None)
    assert call((0.5, 2.0)) == 0
    assert call(None) == -1 and "null" in _err(lib)
    for sp in ((0.0, 1.0), (1.0, float("inf")), (1e-200, 1.0)):
        assert call(sp) == -1 and "spacing" in _err(lib), sp


# ------------------------------------------------------------------------------------------ Python argument checks
def test_spacing_arguments():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    assert derive.spacing_2d(None) is None
    assert derive.spacing_2d((1, 2)) == (1.0, 2.0)
    assert derive.spacing_2d(np.array([0.0039, 0.0117])) == OCT
    for sp in ((1,), (1, 1, 1), (0, 1), (1, -1), (np.nan, 1), (1, np.inf), (1e-300, 1), (1, 1e200), "ab", (1, "x")):
        with pytest.raises(ValueError, match="spacing"):
            derive.spacing_2d(sp)


def test_surface_dice_tolerance_limits():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    assert derive.surface_dice_spacing_limit((1, 1)) == float(np.nextafter(8.5, 0))
    assert derive.surface_dice_spacing_tolerances((8.0, 0.0), (1, 1)) == (8.0, 0.0)
    assert derive.surface_dice_spacing_tolerances(2, (1, 1)) == (2.0,)
    with pytest.raises(ValueError, match=r"largest tolerance allowed is 8\.49999"):
        derive.surface_dice_spacing_tolerances(8.5, (1, 1))
    # rows limit the OCT spacing, columns the transposed one: the limit is the smaller of the two
    lim = derive.surface_dice_spacing_limit(OCT)
    assert lim == float(np.nextafter(np.sqrt(OCT[0] ** 2 * 289 / 4.0), 0))
    assert derive.surface_dice_spacing_limit(OCT[::-1]) == lim
    assert derive.surface_dice_spacing_tolerances(lim, OCT) == (lim,)
    with pytest.raises(ValueError, match="largest tolerance"):
        derive.surface_dice_spacing_tolerances(0.034, OCT)
    for taus in ((), (1, 2, 3, 4, 5)):
        with pytest.raises(ValueError, match="1 to 4"):
            derive.surface_dice_spacing_tolerances(taus, (1, 1))
    for taus in ((-1,), (np.nan,), (np.inf,)):
        with pytest.raises(ValueError, match="finite"):
            derive.surface_dice_spacing_tolerances(taus, (1, 1))
    with pytest.raises(ValueError, match="not a number"):
        derive.surface_dice_spacing_tolerances(("x",), (1, 1))


def test_host_epilogue_scales_by_the_row_spacing():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    thick, bsq, bab, w = np.array([[7, 0]]), np.array([[13]]), np.array([[5]]), 3
    sy = 0.0039
    assert derive.thickness_difference(thick, w, (sy, 0.0117))[0, 0] == (7 / 3) * sy
    b = derive.boundary_errors(bsq, bab, w, (sy, 0.0117))
    assert b["boundary_mse"][0, 0] == (13 / 3) * (sy * sy)
    assert b["boundary_rmse"][0, 0] == np.sqrt((13 / 3) * (sy * sy))
    assert b["boundary_mad"][0, 0] == (5 / 3) * sy
    # a spacing of 1 multiplies by 1.0: the pixel values
    assert np.array_equal(derive.thickness_difference(thick, w, (1, 1)), derive.thickness_difference(thick, w))
    for key, v in derive.boundary_errors(bsq, bab, w, (1.0, 5.0)).items():
        assert np.array_equal(v, derive.boundary_errors(bsq, bab, w)[key]), key


# ------------------------------------------------------------------------------------------ oracle
def _masks():
    rng = np.random.default_rng(2024)
    for _ in range(16):
        h, w = (int(v) for v in rng.integers(2, 11, size=2))
        yield rng.random((h, w)) < rng.uniform(0.2, 0.8), rng.random((h, w)) < rng.uniform(0.2, 0.8)
    yy, xx = np.ogrid[:9, :12]
    disc = (yy - 4) ** 2 + (xx - 6) ** 2 < 10
    yield disc, np.roll(disc, 2, axis=1)
    yield np.zeros((5, 6), bool), np.ones((5, 6), bool)


SPACINGS = ((1.0, 1.0), OCT, OCT[::-1], (1.0, 30.0), (30.0, 1.0), (0.5, 2.0))


@pytest.mark.parametrize("mode", ["first", "all"])
@pytest.mark.parametrize("spacing", SPACINGS)
def test_oracle_against_python_search(mode, spacing):
    seen = 0
    for a, b in _masks():
        im = so.intermediates(a, b, spacing, mode)
        if im is None:
            assert so.vertices(a, mode) is None or so.vertices(b, mode) is None
            continue
        seen += 1
        for key, src, qry in (("sq_pred_to_true", "verts_true", "verts_pred"),
                              ("sq_true_to_pred", "verts_pred", "verts_true")):
            got, want = im[key], so.python_search(im[src], im[qry], spacing)
            assert got.dtype == np.float64 and np.array_equal(got, want), (mode, spacing, key)
    assert seen >= 12


@pytest.mark.parametrize("mode", ["first", "all"])
def test_oracle_unit_spacing_is_the_pixel_oracle(mode):
    for a, b in _masks():
        im = so.intermediates(a, b, (1, 1), mode)
        if im is None:
            continue
        assert np.array_equal(im["sq_pred_to_true"], directed_sq_distances(im["verts_true"], im["verts_pred"]))
        assert np.array_equal(im["sq_true_to_pred"], directed_sq_distances(im["verts_pred"], im["verts_true"]))


def test_anisotropy_changes_the_nearest_vertex():
    """At 30:1 (columns 30 times wider) the source one lattice column away is farther than the one 10 rows away."""
    src = np.array([[0, 1], [10, 0]])
    qry = np.array([[0, 0]])
    assert so.squared_distances(src, qry, (1, 1)).tolist() == [1.0]
    assert so.squared_distances(src, qry, (1, 30)).tolist() == [100.0]
    assert so.order_statistics([4.0, 1.0, 9.0]) == (9.0, 4.0, 9.0)


# ------------------------------------------------------------------------------------------ files
def test_evaluate_files_header_spacing(tmp_path, monkeypatch):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import datasets, suite
    vol = np.zeros((2, 6, 8), np.uint8)
    datasets.write_mhd(str(tmp_path / "t.mhd"), vol, spacing=(0.0117, 0.0039, 0.047))      # header order x, y, z
    datasets.write_mhd(str(tmp_path / "p.mhd"), vol)
    datasets.write_mhd(str(tmp_path / "n.mhd"), vol)
    np.save(tmp_path / "t.npy", vol)
    seen = {}
    monkeypatch.setattr(suite, "evaluate_host", lambda yt, yp, k, **kw: seen.update(kw) or "ok")
    assert datasets.evaluate_files(str(tmp_path / "t.mhd"), str(tmp_path / "p.mhd"), 3, spacing="header") == "ok"
    assert seen["spacing"] == (0.0039, 0.0117)                                             # (rows, cols)
    assert datasets.evaluate_files(str(tmp_path / "t.mhd"), str(tmp_path / "p.mhd"), 3) == "ok"
    assert seen["spacing"] is None
    with pytest.raises(ValueError, match="ElementSpacing"):
        datasets.evaluate_files(str(tmp_path / "n.mhd"), str(tmp_path / "p.mhd"), 3, spacing="header")
    with pytest.raises(ValueError, match="MetaImage"):
        datasets.evaluate_files(str(tmp_path / "t.npy"), str(tmp_path / "t.npy"), 3, spacing="header")
    with pytest.raises(ValueError, match="header"):
        datasets.evaluate_files(str(tmp_path / "t.mhd"), str(tmp_path / "p.mhd"), 3, spacing="rows")


# ------------------------------------------------------------------------------------------ dataset totals (gloo)
K, W = 4, 16


def _vec(rank):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    rng = np.random.default_rng(rank + 5)
    vec = np.zeros(odist.base_len(K))
    vec[0] = 3
    vec[1:] = rng.integers(0, 50, size=len(vec) - 1)
    vec[-2:] = 0                                      # no overflow, no bad labels
    return vec


def _worker(rank, world, port, q):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
    vec = odist.all_reduce_sum(_vec(rank), world, device="cpu")
    q.put((rank, {key: v for key, v in odist.unpack(vec, K, W, OCT).items()}))
    torch.distributed.destroy_process_group()


def test_unpack_scales_dataset_means_by_the_spacing():
    import torch.multiprocessing as mp
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    total = _vec(0) + _vec(1)
    plain = odist.unpack(total, K, W)
    sy = OCT[0]
    for r in range(2):
        out = got[r]
        assert np.array_equal(out["thickness_difference"], plain["thickness_difference"] * sy)
        assert np.array_equal(out["boundary_mse"], plain["boundary_mse"] * (sy * sy))
        assert np.array_equal(out["boundary_rmse"], np.sqrt(plain["boundary_mse"] * (sy * sy)))
        assert np.array_equal(out["boundary_mad"], plain["boundary_mad"] * sy)
        for key in ("confusion", "dice_coefficient", "contour_items"):
            assert np.array_equal(out[key], plain[key], equal_nan=True), key
    unit = odist.unpack(total, K, W, (1.0, 1.0))
    for key in plain:
        assert np.array_equal(np.asarray(unit[key]), np.asarray(plain[key]), equal_nan=True), key
