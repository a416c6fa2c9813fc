"""CPU tier: octm_surface3d_spacing_u8 validates its arguments before any CUDA call, the spacing oracle agrees with a
brute-force search, and the host-side pieces (argument checks, floating squared distances in derive, MetaImage
spacing) behave."""
import ctypes

import numpy as np
import pytest

import surface3d_spacing_oracle as sso
from oracle import surface3d_oracle as s3


@pytest.fixture(scope="module")
def lib():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails
OUTS = ("y_true", "y_pred", "n_pts", "max_sq", "p95_sq", "sum_dist", "n_surf", "n_within")


def _call(lib, shape=(8, 8, 16), k=2, units=None, spacing=(1.0, 1.0, 1.0), taus=(1.0,), ntau=None, null=(),
          ws_bytes=0):
    """``null`` names the pointers passed as NULL (also "spacing" and "tolerances").  The workspace is too small by
    default, so a call that passes every other check returns OCTM_ERR_WORKSPACE (-4), still before any CUDA call."""
    p = {name: None if name in null else FAKE for name in OUTS}
    ub, ue = (0, 2 * k) if units is None else units
    sp = None if "spacing" in null else (ctypes.c_double * 3)(*spacing)
    tol = None if "tolerances" in null else (ctypes.c_double * max(1, len(taus)))(*taus)
    return lib.octm_surface3d_spacing_u8(p["y_true"], p["y_pred"], *shape, k, ub, ue, sp, tol,
                                         len(taus) if ntau is None else ntau, p["n_pts"], p["max_sq"], p["p95_sq"],
                                         p["sum_dist"], p["n_surf"], p["n_within"], FAKE, ws_bytes, None)


def _err(lib):
    return lib.octm_last_error().decode()


def test_shape_classes_units_and_sides(lib):
    for shape in ((0, 8, 16), (8, 0, 16), (8, 8, 0), (-1, 8, 16)):
        assert _call(lib, shape) == -1 and "shape" in _err(lib), shape
    for k in (0, 257):
        assert _call(lib, k=k, units=(0, 0)) == -1 and "num_classes" in _err(lib), k
    for units in ((-1, 4), (0, 5), (3, 2)):
        assert _call(lib, units=units) == -1 and "unit range" in _err(lib), units
    for shape in ((2049, 8, 16), (8, 2049, 16), (8, 8, 65535)):
        assert _call(lib, shape) == -2 and "volume sides" in _err(lib), shape
    # no histogram: a squared diagonal beyond 2^28 voxels^2 is fine here (octm_surface3d_u8 refuses it)
    for shape in ((2048, 2048, 16384), (2048, 8, 16), (8, 2048, 65534)):
        assert _call(lib, shape) == -4, shape
    assert _call(lib, k=256) == -4


def test_bad_spacing(lib):
    for sp in ((0.0, 1.0, 1.0), (1.0, -0.5, 1.0), (1.0, 1.0, float("nan")), (float("inf"), 1.0, 1.0),
               (1.0, 1.0, -float("inf")), (1.0, -0.0, 1.0)):
        assert _call(lib, spacing=sp) == -1, sp
        assert "spacing" in _err(lib), sp
    assert _call(lib, spacing=(0.0039, 0.0117, 0.047)) == -4
    # finite and > 0, but the square overflows to inf or underflows to 0 / a subnormal
    for sp in ((1e-300, 1.0, 1.0), (1.0, 1e300, 1.0), (1.0, 1.0, 5e-324), (1.0, 1.0, 1.4e154), (1e-155, 1.0, 1.0)):
        assert _call(lib, spacing=sp) == -1, sp
        assert "square" in _err(lib), sp
    # every square normal, but the squared diagonal of the volume overflows
    assert _call(lib, shape=(8, 8, 16), spacing=(1.0, 1.0, 1.3e154)) == -1 and "diagonal" in _err(lib)
    assert _call(lib, spacing=(1e-150, 1e150, 1.0)) == -4              # tiny and huge, squares and diagonal finite


def test_bad_tolerances(lib):
    assert _call(lib, taus=(1.0, 2.0, 3.0, 4.0, 5.0)) == -1 and "num_tolerances" in _err(lib)
    assert _call(lib, taus=(1.0,), ntau=-1) == -1 and "num_tolerances" in _err(lib)
    for taus in ((float("nan"),), (1.0, -0.1), (float("inf"),), (0.5, 1.0, -float("inf"))):
        assert _call(lib, taus=taus) == -1, taus
        assert "tolerances[" in _err(lib), taus
    for taus in ((0.0,), (0.0, 0.5, 1e9, 2.0)):
        assert _call(lib, taus=taus) == -4, taus
    assert _call(lib, taus=()) == -4                                   # no tolerances: distances only


def test_null_pointers(lib):
    for name in ("y_true", "y_pred", "n_pts", "max_sq", "p95_sq", "sum_dist", "spacing"):
        assert _call(lib, null=(name,)) == -1, name
        assert "null" in _err(lib), name
    for name in ("n_surf", "n_within", "tolerances"):
        assert _call(lib, null=(name,)) == -1, name                      # needed with tolerances
        assert "null" in _err(lib), name
        assert _call(lib, taus=(), null=(name,)) == -4, name             # not needed without


def test_workspace(lib):
    need = lib.octm_surface3d_spacing_workspace_bytes(8, 8, 16)
    assert need >= 8 * 8 * 16 * (8 + 8)                                  # h2 and the query values, float64 per voxel
    assert _call(lib, ws_bytes=need - 1) == -4 and "workspace" in _err(lib)
    rc = lib.octm_surface3d_spacing_u8(FAKE, FAKE, 8, 8, 16, 2, 0, 4, (ctypes.c_double * 3)(1, 1, 1), None, 0, FAKE,
                                       FAKE, FAKE, FAKE, None, None, None, need, None)
    assert rc == -4                                                      # null workspace
    for shape in ((0, 8, 16), (8, 0, 16), (8, 8, 0), (-3, 8, 16)):
        assert lib.octm_surface3d_spacing_workspace_bytes(*shape) == 0, shape
    assert lib.octm_surface3d_spacing_workspace_bytes(1, 1, 1) > 0


# ------------------------------------------------------------------------------------------ oracle vs brute force
def _brute_squared_distances(mask_from, mask_to, spacing):
    pa, pb = np.argwhere(s3.surface(mask_from)), np.argwhere(s3.surface(mask_to))
    if len(pa) == 0 or len(pb) == 0:
        return None
    off = (pa[:, None, :] - pb[None, :, :]).reshape(-1, 3)
    return sso.d2_of_offsets(off, spacing).reshape(len(pa), len(pb)).min(1)


def _volumes():
    rng = np.random.default_rng(71)
    for _ in range(24):
        shape = tuple(int(s) for s in rng.integers(1, 12, size=3))
        yield rng.random(shape) < rng.uniform(0.05, 0.9), rng.random(shape) < rng.uniform(0.05, 0.9)
    full = np.ones((5, 6, 7), bool)
    yield np.zeros_like(full), full
    yield full, np.zeros_like(full)


DYADIC = ((0.5, 1.0, 2.0), (1.0, 1.0, 4.0), (0.25, 3.0, 1.0))
OCT_LIKE = ((0.0039, 0.0117, 0.047), (0.047, 0.0039, 0.0117), (1.0, 1.0, 30.0))


@pytest.mark.parametrize("spacing", DYADIC + OCT_LIKE)
def test_oracle_against_brute_force(spacing):
    seen = 0
    for a, b in _volumes():
        got, want = sso.squared_distances(a, b, spacing), _brute_squared_distances(a, b, spacing)
        if want is None:
            assert got is None, a.shape
            continue
        seen += 1
        assert got.dtype == np.float64
        if spacing in DYADIC:                      # every product and sum is exact: scipy's choice is the minimum
            assert np.array_equal(got, want), a.shape
        else:                                      # ties broken by scipy's own rounding: a few ulp at most
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert seen >= 20


def test_oracle_unit_spacing_is_the_voxel_oracle():
    for a, b in _volumes():
        got, want = sso.squared_distances(a, b, (1, 1, 1)), s3.squared_distances(a, b)
        assert (got is None) == (want is None)
        if want is not None:
            assert np.array_equal(got, want.astype(np.float64))


def test_oracle_anisotropy_changes_the_nearest_voxel():
    """30:1 along D2: the source voxel one step along D2 is farther than the one 5 steps along D0."""
    a = np.zeros((12, 3, 4), bool)
    b = np.zeros((12, 3, 4), bool)
    a[0, 1, 1] = True
    b[0, 1, 2] = True                              # one step along D2
    b[5, 1, 1] = True                              # five steps along D0
    assert sso.squared_distances(a, b, (1, 1, 1)).tolist() == [1.0]
    assert sso.squared_distances(a, b, (1, 1, 30)).tolist() == [25.0]


# ------------------------------------------------------------------------------------------ host-side pieces
def test_spacing_arguments():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    assert suite.surface3d_spacing_args(None, None) == ((1.0, 1.0, 1.0), ())
    assert suite.surface3d_spacing_args(None, 2) == ((1.0, 1.0, 1.0), (2.0,))
    assert suite.surface3d_spacing_args(np.array([0.5, 1, 2]), (0, 100.0)) == ((0.5, 1.0, 2.0), (0.0, 100.0))
    for sp in ((1, 1), (1, 1, 1, 1), (0, 1, 1), (1, -1, 1), (1, 1, np.nan), (np.inf, 1, 1), (1e-300, 1, 1),
               (1, 1e200, 1), (1, 1, 5e-324)):
        with pytest.raises(ValueError, match="spacing"):
            suite.surface3d_spacing_args(sp, None)
    assert suite.surface3d_spacing_args((1e-150, 1e150, 1), None) == ((1e-150, 1e150, 1.0), ())
    for taus in ((), (1, 2, 3, 4, 5)):
        with pytest.raises(ValueError, match="tolerances"):
            suite.surface3d_spacing_args(None, taus)
    for taus in ((-1,), (np.nan,), (1, np.inf)):
        with pytest.raises(ValueError, match="tolerances"):
            suite.surface3d_spacing_args((1, 1, 1), taus)
    assert suite.surface3d_spacing_args(None, (9.0, 50.0)) == ((1.0, 1.0, 1.0), (9.0, 50.0))   # no 8-voxel cap


def test_contour_metrics_keep_floating_squared_distances():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import derive
    n_pts = np.array([[3, 4]])
    max_sq = np.array([[2.25, 0.5]])
    p95 = np.array([[[0.5, 2.25], [0.25, 0.5]]])
    sums = np.array([[2.0, 3.0]])
    m = derive.contour_metrics(n_pts, max_sq, p95, sums, lattice=1.0)
    assert m["hausdorff_distance"][0] == 1.5                         # sqrt(2.25); truncation would give 1.414
    # lists with those order statistics: direction 0 has 4 query voxels (n_pts[1]), direction 1 has 3
    d0, d1 = np.sqrt([0.125, 0.25, 0.5, 2.25]), np.sqrt([0.125, 0.25, 0.5])
    want = max(np.percentile(d0, 95), np.percentile(d1, 95))
    np.testing.assert_allclose(m["hausdorff_distance_95"][0], want, rtol=1e-12)
    ints = derive.contour_metrics(n_pts, np.array([[2, 1]], np.uint32), np.array([[[1, 2], [1, 1]]], np.uint32), sums,
                                  lattice=1.0)
    assert ints["hausdorff_distance"][0] == np.sqrt(2.0)             # integer inputs as before


def test_mhd_spacing(tmp_path):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import datasets
    vol = np.arange(2 * 3 * 4, dtype=np.uint8).reshape(2, 3, 4)
    for compressed in (False, True):
        p = tmp_path / f"v{int(compressed)}.mhd"
        datasets.write_mhd(str(p), vol, spacing=(0.0117, 0.0039, 0.047), compressed=compressed)   # header order x, y, z
        arr, header = datasets.read_mhd(str(p))
        assert arr.shape == (2, 3, 4)
        assert datasets.mhd_spacing(header) == (0.047, 0.0039, 0.0117)                          # array axes z, y, x
    with pytest.raises(KeyError, match="ElementSpacing"):
        datasets.write_mhd(str(tmp_path / "n.mhd"), vol)
        datasets.mhd_spacing(datasets.read_mhd(str(tmp_path / "n.mhd"))[1])
    with pytest.raises(ValueError, match="entries"):
        datasets.mhd_spacing({"NDims": "3", "ElementSpacing": "1 1"})
    with pytest.raises(ValueError, match="numbers"):
        datasets.mhd_spacing({"NDims": "3", "ElementSpacing": "1 a 1"})


# ------------------------------------------------------------------------------------------ sharded packing (gloo)
K_SHARD = 3


def _fake_units(vol_true, vol_pred, num_classes, *, units, spacing=None, tolerances=None):
    """Stand-in for suite.surface_distance_3d on the CPU: every unit in ``units`` writes its own entries only, with
    values that a float64 round trip must keep (non-integral squared distances, uint32 counts above 2**31)."""
    import torch
    k = num_classes
    f64 = spacing is not None or tolerances is not None
    sq = torch.float64 if f64 else torch.int32
    out = {"n_pts": torch.zeros((k, 2), dtype=torch.int32), "max_sq": torch.zeros((k, 2), dtype=sq),
           "p95_sq": torch.zeros((k, 2, 2), dtype=sq), "sum_dist": torch.zeros((k, 2), dtype=torch.float64)}
    if tolerances is not None:
        out["n_surf"] = torch.zeros((k, 2), dtype=torch.int32)
        out["n_within"] = torch.zeros((k, 2, len(tolerances)), dtype=torch.int32)
    for u in range(*units):
        c, d = divmod(u, 2)
        out["n_pts"][c, 1 - d] = -7 - u                                  # uint32 4294967289 - u
        out["max_sq"][c, d] = (u + 1) / 3 if f64 else -2 - u            # uint32 above 2**31
        out["p95_sq"][c, d] = torch.tensor([u / 7, u / 5] if f64 else [u, -u - 1]).to(sq)
        out["sum_dist"][c, d] = u / 11 + 1e-9
        if tolerances is not None:
            out["n_surf"][c, 1 - d] = 100 + u
            out["n_within"][c, d] = torch.arange(len(tolerances), dtype=torch.int32) + u
    return out


def _shard_worker(rank, world, port, q):
    import os
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
    suite.surface_distance_3d = _fake_units
    got = []
    for kw in ({}, {"spacing": (0.5, 1, 2)}, {"spacing": (0.5, 1, 2), "tolerances": (0.1, 0.2)}):
        # numpy arrays travel by value: a torch tensor would be shared through a file descriptor of this process,
        # which may have exited by the time the parent unpickles it
        got.append({key: v.numpy().copy() for key, v in odist.surface_distance_3d_sharded(None, None, K_SHARD, rank,
                                                                                             world, **kw).items()})
    q.put((rank, got))
    torch.distributed.destroy_process_group()


def test_sharded_outputs_equal_the_unsharded_ones():
    """Two ranks (gloo): the single all-reduce returns every unit's entries bit for bit, dtypes and shapes as the
    unsharded call, on the integer path, with a spacing and with tolerances."""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    for i, kw in enumerate(({}, {"spacing": (0.5, 1, 2)}, {"spacing": (0.5, 1, 2), "tolerances": (0.1, 0.2)})):
        want = _fake_units(None, None, K_SHARD, units=(0, 2 * K_SHARD), **kw)
        for r in range(2):
            assert list(got[r][i]) == list(want), (r, kw)
            for key in want:
                w = want[key].numpy()
                assert got[r][i][key].dtype == w.dtype and np.array_equal(got[r][i][key], w), (r, kw, key)
