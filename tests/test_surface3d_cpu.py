"""CPU tier: octm_surface3d_u8 validates its arguments before any CUDA call, and the 3-D surface-distance oracle agrees
with brute force."""
import ctypes

import numpy as np
import pytest

from oracle import surface3d_oracle as s3


@pytest.fixture(scope="module")
def lib():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails


def _call(lib, shape=(8, 8, 16), k=2, units=None, null=(), ws_bytes=0):
    """``null`` names the pointers passed as NULL.  The workspace is too small by default, so a call that passes every
    other check returns OCTM_ERR_WORKSPACE (-4), still before any CUDA call."""
    p = {name: None if name in null else FAKE for name in ("y_true", "y_pred", "n_pts", "max_sq", "p95_sq", "sum_dist")}
    ub, ue = (0, 2 * k) if units is None else units
    return lib.octm_surface3d_u8(p["y_true"], p["y_pred"], *shape, k, ub, ue, p["n_pts"], p["max_sq"], p["p95_sq"],
                                 p["sum_dist"], FAKE, ws_bytes, None)


def test_bad_shape(lib):
    for shape in ((0, 8, 16), (8, 0, 16), (8, 8, 0), (-1, 8, 16)):
        assert _call(lib, shape) == -1, shape
        assert b"shape" in lib.octm_last_error()


def test_bad_num_classes(lib):
    for k in (0, 257):
        assert _call(lib, k=k, units=(0, 0)) == -1, k
        assert b"num_classes" in lib.octm_last_error()
    assert _call(lib, k=256) == -4                                      # 256 classes pass the class check


def test_bad_unit_range(lib):
    for units in ((-1, 4), (0, 5), (3, 2)):
        assert _call(lib, k=2, units=units) == -1, units
        assert b"unit range" in lib.octm_last_error()
    for units in ((0, 4), (4, 4), (1, 2)):
        assert _call(lib, k=2, units=units) == -4, units


def test_null_pointers(lib):
    for name in ("y_true", "y_pred", "n_pts", "max_sq", "p95_sq", "sum_dist"):
        assert _call(lib, null=(name,)) == -1, name
        assert b"null" in lib.octm_last_error()


def test_unsupported_sizes(lib):
    for shape in ((2049, 8, 16), (8, 2049, 16), (8, 8, 65535)):
        assert _call(lib, shape) == -2, shape
        assert b"volume sides" in lib.octm_last_error()
    # 2047^2 + 2047^2 + 16383^2 >= 2^28: the histogram of squared distances would be too large
    assert _call(lib, (2048, 2048, 16384)) == -2
    assert b"squared diagonal" in lib.octm_last_error()
    for shape in ((2048, 8, 16), (8, 2048, 16), (2048, 2048, 16)):
        assert _call(lib, shape) == -4, shape


def test_workspace_too_small(lib):
    need = lib.octm_surface3d_workspace_bytes(8, 8, 16)
    assert need >= 8 * 8 * 16 * (2 + 4)                                 # g (uint16) and h2 (uint32) per voxel at least
    assert _call(lib, ws_bytes=need - 1) == -4
    assert b"workspace" in lib.octm_last_error()
    assert _call(lib, k=256, ws_bytes=need - 1) == -4
    rc = lib.octm_surface3d_u8(FAKE, FAKE, 8, 8, 16, 2, 0, 4, FAKE, FAKE, FAKE, FAKE, None, need, None)
    assert rc == -4                                                     # null workspace


def test_workspace_bytes_of_an_empty_shape(lib):
    for shape in ((0, 8, 16), (8, 0, 16), (8, 8, 0), (-3, 8, 16)):
        assert lib.octm_surface3d_workspace_bytes(*shape) == 0, shape
    assert lib.octm_surface3d_workspace_bytes(1, 1, 1) > 0


# ------------------------------------------------------------------------------------------ oracle vs brute force
def _brute_surface(mask):
    """Voxels of the mask with one of their six neighbours outside it; outside the volume counts as outside."""
    pad = np.pad(mask, 1)
    out = np.zeros_like(mask)
    for idx in np.argwhere(mask):
        i, j, k = idx + 1
        out[tuple(idx)] = not (pad[i - 1, j, k] and pad[i + 1, j, k] and pad[i, j - 1, k] and pad[i, j + 1, k] and
                               pad[i, j, k - 1] and pad[i, j, k + 1])
    return out


def _brute_squared_distances(mask_from, mask_to):
    pa, pb = np.argwhere(_brute_surface(mask_from)), np.argwhere(_brute_surface(mask_to))
    if len(pa) == 0 or len(pb) == 0:
        return None
    return ((pa[:, None, :] - pb[None, :, :]) ** 2).sum(-1).min(1)


def _volumes():
    rng = np.random.default_rng(61)
    for _ in range(30):
        shape = tuple(int(s) for s in rng.integers(1, 14, size=3))
        yield rng.random(shape) < rng.uniform(0.05, 0.9), rng.random(shape) < rng.uniform(0.05, 0.9)
    for shape in ((1, 1, 1), (1, 1, 40), (7, 9, 1), (1, 30, 1), (12, 1, 10)):
        yield rng.random(shape) < 0.3, rng.random(shape) < 0.3
    full = np.ones((6, 7, 8), bool)                                     # a full volume: its surface is the border
    yield full, full
    yield np.zeros_like(full), full                                     # an empty surface on either side
    yield full, np.zeros_like(full)


def test_oracle_against_brute_force():
    seen_none = seen_values = 0
    for a, b in _volumes():
        sa, sb = s3.surface(a), s3.surface(b)
        assert np.array_equal(sa, _brute_surface(a)) and np.array_equal(sb, _brute_surface(b)), a.shape
        got, want = s3.squared_distances(a, b), _brute_squared_distances(a, b)
        if want is None:
            assert got is None, a.shape
            seen_none += 1
        else:
            assert got is not None and got.dtype == np.int64 and np.array_equal(got, want), a.shape
            seen_values += 1
    assert seen_none >= 2 and seen_values >= 30
