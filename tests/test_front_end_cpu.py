"""CPU checks of ``suite._raster_rows``, the host conversion in front of the rasterise kernel
(``suite.labels_from_boundaries``).  The kernel reads float32 or int32 rows; the conversion must keep, for every row
``y`` of a map, whether ``b <= y`` holds on the caller's own values, float64 and int64 included."""
import numpy as np
import pytest
import torch

from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite

NEVER = 2**31 - 1

F64_EDGES = [np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-50, -1e-50, 5e-324, -5e-324, 1e-300, 0.5, -0.5, 1.0, -1.0,
             99.9999999, 100.0, 100.0000001, 100 + 2**-20, 100 - 2**-20, 4097 + 2**-20, 2**31 - 1.5, 2**31 - 1.0,
             2**31 - 0.5, 2.0**31, 2**31 + 0.5, -(2**31) + 0.5, -(2.0**31), -(2**31) - 0.5, -(2**31) - 10.0, 3e9, -3e9,
             1e300, -1e300, np.finfo(np.float64).max, -np.finfo(np.float64).max]
I64_EDGES = [0, -1, 1, 5, 99, 100, 101, NEVER - 1, NEVER, 2**31, 2**32 + 5, 2**32 - 1, -(2**31) + 1, -(2**31),
             -(2**31) - 10, -(2**32) + 5, 2**63 - 1, -(2**63)]


def _ref(values):
    """The int32 threshold of each value: ceil, NaN -> never, clamped to [-(2**31 - 1), 2**31 - 1]."""
    v = np.asarray(values, dtype=np.float64)
    return np.clip(np.where(np.isnan(v), NEVER, np.ceil(v)), -NEVER, NEVER).astype(np.int32)


def test_float64_rows_become_clamped_ceilings():
    b = torch.tensor(F64_EDGES, dtype=torch.float64)
    got, dt = suite._raster_rows(b)
    assert dt == _lib.DTYPE_I32 and got.dtype == torch.int32
    np.testing.assert_array_equal(got.numpy(), _ref(F64_EDGES))
    assert got[F64_EDGES.index(100.0000001)] == 101 and got[F64_EDGES.index(1e-50)] == 1
    assert got[F64_EDGES.index(-1e-50)] == 0 and got[0] == NEVER and got[2] == -NEVER


@pytest.mark.parametrize("dtype", [torch.int64, torch.uint32, torch.uint64])
def test_wide_integer_rows_are_clamped(dtype):
    info = torch.iinfo(dtype)
    vals = [v for v in I64_EDGES if info.min <= v <= info.max]
    if dtype == torch.uint64:
        vals += [2**63, 2**64 - 1]
        b = torch.tensor(np.array(vals, dtype=np.uint64))
    else:
        b = torch.tensor(vals, dtype=torch.int64).to(dtype)
    got, dt = suite._raster_rows(b)
    assert dt == _lib.DTYPE_I32 and got.dtype == torch.int32
    want = [min(max(v, -NEVER), NEVER) for v in vals]
    assert got.tolist() == want


@pytest.mark.parametrize("dtype", [torch.bool, torch.int8, torch.uint8, torch.int16, torch.uint16, torch.int32])
def test_narrow_integer_rows_pass_as_int32(dtype):
    if dtype == torch.bool:
        vals = [0, 1]
    else:
        info = torch.iinfo(dtype)
        vals = sorted({info.min, info.min + 1, min(info.min + 2, 0), 0, 1, info.max})
    b = torch.tensor(vals, dtype=torch.int64).to(dtype)
    got, dt = suite._raster_rows(b)
    assert dt == _lib.DTYPE_I32 and got.dtype == torch.int32
    assert got.tolist() == [int(v) for v in vals]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32])
def test_narrow_float_rows_pass_exactly_as_float32(dtype):
    fi = torch.finfo(dtype)
    vals = [np.nan, np.inf, -np.inf, 0.0, -0.0, fi.max, -fi.max, fi.tiny, fi.smallest_normal / 4, -fi.smallest_normal / 4,
            fi.eps, 1 + fi.eps, 2.5, -7.0, 100.0 + 2**-3]
    b = torch.tensor(vals, dtype=torch.float64).to(dtype)
    got, dt = suite._raster_rows(b)
    assert dt == _lib.DTYPE_F32 and got.dtype == torch.float32
    want = b.to(torch.float64).numpy()
    assert np.array_equal(got.to(torch.float64).numpy(), want, equal_nan=True)
    assert np.signbit(got.numpy()[4])                               # -0.0 stays -0.0


def test_converted_rows_rasterise_like_the_originals():
    """The oracle on the converted int32 rows equals the oracle on the caller's float64 / int64 rows, for every row of
    a map; the float32 / int32 narrowing this replaces does not."""
    h = 130
    f = np.array(F64_EDGES, dtype=np.float64)
    i = np.array(I64_EDGES, dtype=np.int64)
    for rows in (f, i):
        b = rows.reshape(1, 1, -1)
        want = lo.labels_from_boundaries(b, h)
        got = lo.labels_from_boundaries(suite._raster_rows(torch.from_numpy(b))[0].numpy(), h)
        np.testing.assert_array_equal(got, want)
    with np.errstate(over="ignore"):
        narrowed_f = lo.labels_from_boundaries(f.astype(np.float32).reshape(1, 1, -1), h)
    narrowed_i = lo.labels_from_boundaries(i.astype(np.int32).reshape(1, 1, -1), h)
    assert not np.array_equal(narrowed_f, lo.labels_from_boundaries(f.reshape(1, 1, -1), h))
    assert not np.array_equal(narrowed_i, lo.labels_from_boundaries(i.reshape(1, 1, -1), h))


def test_conversion_keeps_shape_and_is_contiguous():
    b = torch.arange(24, dtype=torch.float64).reshape(2, 3, 4).transpose(1, 2) + 0.25
    got, _ = suite._raster_rows(b)
    assert got.shape == b.shape and got.is_contiguous()
    np.testing.assert_array_equal(got.numpy(), np.ceil(b.numpy()).astype(np.int32))
