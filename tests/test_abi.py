"""CPU tier: the C-ABI library loads without a GPU and exports exactly what include/octm.h declares."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib


def _header_decls():
    src = open(os.path.join(ROOT, "include", "octm.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    decls = {}
    for m in re.finditer(r"OCTM_API\s+([\w\s\*]+?)\s*\b(octm_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(3).strip()
        n = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
        decls[m.group(2)] = n
    return decls


def test_every_declared_symbol_is_exported_and_bound(lib):
    decls = _header_decls()
    assert len(decls) >= 14
    so = lib.load()
    out = subprocess.run(["nm", "-D", "--defined-only", lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (octm_\w+)", out))
    assert set(decls) == exported, (set(decls) ^ exported)
    assert set(decls) == set(lib.SIGNATURES)
    for name, nargs in decls.items():
        assert len(lib.SIGNATURES[name][1]) == nargs, name
        assert getattr(so, name) is not None


def test_abi_version_and_error_channel(lib):
    so = lib.load()
    assert so.octm_abi_version() == 1
    # argument validation happens before any CUDA call, so it works without a GPU
    rc = so.octm_confusion_u8(None, None, 1, 16, 99, None, None)
    assert rc == -1 and b"num_classes" in so.octm_last_error()
    rc = so.octm_label_pass_u8(None, None, -1, 4, 4, 2, None, None, None, None, None, None, None, None)
    assert rc == -1
    assert so.octm_contour2d_workspace_bytes(10, 496, 512, 8, 2048) >= 10 * 8 * 2 * 2048 * 4


def test_fast_path_predicate(lib):
    so = lib.load()
    assert so.octm_label_pass_path(496, 512, 8, 0, 0) == 1
    assert so.octm_label_pass_path(496, 768, 8, 0, 0) == 1
    assert so.octm_label_pass_path(496, 1024, 10, 0, 0) == 2      # K > 8 -> warp-per-strip run-length kernel (K <= 16, W % 4 == 0)
    assert so.octm_label_pass_path(496, 500, 8, 0, 0) == 2        # W % 16 != 0 but W % 4 == 0
    assert so.octm_label_pass_path(33, 50, 4, 0, 0) == 0          # ragged width -> byte-wise generic kernel
    assert so.octm_label_pass_path(496, 512, 8, 8, 0) == 2        # 8-byte aligned only: not the TMA kernel
    assert so.octm_label_pass_path(496, 512, 8, 1, 0) == 0        # misaligned pointer


def test_sass_uses_tma_tile_copies(lib):
    """The staged label pass must really be TMA: UTMALDG (2-D tensor-map tile loads) in the sm_100a SASS."""
    r = subprocess.run(["cuobjdump", "-sass", lib.LIB_PATH], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in r.stdout or "SM100a" in r.stdout or "sm_100" in r.stdout
    assert "UTMALDG" in r.stdout
    assert "LDG.E.NA.EFL2.256" in r.stdout or ".256" in r.stdout      # 256-bit streaming loads of the argmax front end
    assert "SYNCS" in r.stdout        # mbarrier arrive / try_wait


def test_host_nibble_packer(lib):
    """octm_host_pack_nibbles is a host function (transfer encoding): exercised here without a GPU."""
    import numpy as np
    so = lib.load()
    rng = np.random.default_rng(0)
    for n in (0, 1, 2, 63, 64, 65, 100003, 1 << 21):
        src = rng.integers(0, 16, n, dtype=np.uint8)
        dst = np.full((n + 1) // 2 + 8, 0xAA, np.uint8)
        assert so.octm_host_pack_nibbles(src.ctypes.data, dst.ctypes.data, n, 3) == 0
        ref = np.zeros((n + 1) // 2, np.uint8)
        ref[:n // 2] = src[0:n - (n & 1):2] | (src[1::2] << 4)
        if n & 1:
            ref[-1] = src[-1]
        assert np.array_equal(dst[:(n + 1) // 2], ref) and (dst[(n + 1) // 2:] == 0xAA).all()

    # A label >= 16 has no 4-bit code: the packer must say so (OCTM_PACK_WIDE_LABEL = 1) wherever it sits, in the
    # AVX2 body (64-label blocks), the scalar tail, the odd last label, and in the chunk of any thread (3 threads,
    # at least 64 Ki labels each).
    n = 3 * (1 << 17) + 37
    base = rng.integers(0, 16, n, dtype=np.uint8)
    dst = np.empty((n + 1) // 2, np.uint8)
    assert so.octm_host_pack_nibbles(base.ctypes.data, dst.ctypes.data, n, 3) == 0
    tail = n - (n & 1) - (n - (n & 1)) % 64          # first label of the last thread's scalar tail
    for at in (0, 1, 62, 63, 1 << 17, (1 << 17) + 5, 2 << 17, 3 << 17, tail, tail + 1, n - 2, n - 1):
        for bad in (16, 17, 128, 255):
            src = base.copy()
            src[at] = bad
            assert so.octm_host_pack_nibbles(src.ctypes.data, dst.ctypes.data, n, 3) == 1, (at, bad)
            assert so.octm_host_pack_nibbles(src.ctypes.data, dst.ctypes.data, n, 1) == 1, (at, bad)
    for n in (1, 2, 3, 64, 65):                      # scalar only, one AVX2 block, a block and a tail
        for at in range(n):
            src = np.zeros(n, np.uint8)
            src[at] = 16
            assert so.octm_host_pack_nibbles(src.ctypes.data, dst.ctypes.data, n, 0) == 1, (n, at)
