"""CPU tier: the all-contour entry points validate their arguments before any CUDA call."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def so():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails


def _vertices(so, *, n=1, h=8, w=8, k=2, max_pts=64, ptr=FAKE):
    return so.octm_contour2d_all_vertices_u8(ptr, ptr, n, h, w, k, max_pts, ptr, ptr, ptr, None)


def _all(so, *, n=1, h=8, w=8, k=2, max_pts=64, ptr=FAKE, ws_bytes=1 << 30):
    return so.octm_contour2d_all_u8(ptr, ptr, n, h, w, k, max_pts, ptr, ptr, ptr, ptr, ptr, ptr, ws_bytes, None)


def test_bad_num_classes(so):
    assert _vertices(so, k=99) == -1 and b"num_classes" in so.octm_last_error()
    assert _all(so, k=99) == -1
    assert _vertices(so, k=1) == -1


def test_max_pts_must_be_a_multiple_of_four(so):
    assert _vertices(so, max_pts=10) == -1 and b"max_pts" in so.octm_last_error()
    assert _all(so, max_pts=10) == -1
    assert _vertices(so, max_pts=4) == -1


def test_bad_shape(so):
    assert _vertices(so, n=-1) == -1
    assert _vertices(so, h=0) == -1
    assert _all(so, w=9000) == -2


def test_null_pointers(so):
    assert _vertices(so, ptr=None) == -1 and b"null" in so.octm_last_error()
    assert _all(so, ptr=None) == -1
    rc = so.octm_contour2d_all_vertices_u8(FAKE, None, 1, 8, 8, 2, 64, FAKE, FAKE, FAKE, None)
    assert rc == -1


def test_workspace_too_small(so):
    need = so.octm_contour2d_workspace_bytes(3, 8, 8, 2, 64)
    assert need >= 2 * 3 * 2 * 2 * 64 * 4
    assert _all(so, n=3, ws_bytes=need - 1) == -4 and b"workspace" in so.octm_last_error()
    rc = so.octm_contour2d_all_u8(FAKE, FAKE, 3, 8, 8, 2, 64, FAKE, FAKE, FAKE, FAKE, FAKE, None, need, None)
    assert rc == -4


def test_empty_batch_is_a_no_op(so):
    assert _vertices(so, n=0, ptr=None) == 0
    assert _all(so, n=0, ptr=None, ws_bytes=0) == 0
