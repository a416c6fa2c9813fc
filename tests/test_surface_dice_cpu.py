"""CPU tier of the normalized surface Dice: tolerance thresholds, the NSD ratio, the oracle, argument validation of
octm_surface_dice_u8 and the multi-rank dataset view."""
import ctypes
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, synth
from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
import all_contours_oracle as ao
import surface_dice_oracle as so_

BOUNDARY_TAUS = (0.0, np.sqrt(2) / 2, 1.0, np.sqrt(5) / 2, 8.0)


def _brute_threshold(tau):
    return max(d for d in range(0, 4 * 300) if np.sqrt(d / 4.0) <= tau)


def test_threshold_equals_brute_force_scan():
    taus = []
    for t in BOUNDARY_TAUS + (0.5, 1.5, 2.0, 3.0, 4.0, np.sqrt(10) / 2, np.sqrt(254) / 2, np.sqrt(258) / 4):
        taus += [t, np.nextafter(t, np.inf), np.nextafter(t, -np.inf)]
    taus += list(np.random.default_rng(3).uniform(0, 8, 200))
    for t in taus:
        if t < 0:
            continue
        assert derive.surface_dice_threshold(t) == _brute_threshold(t), t
    assert [derive.surface_dice_threshold(t) for t in BOUNDARY_TAUS] == [0, 2, 4, 5, 256]
    assert derive.surface_dice_threshold(np.nextafter(8.0, -np.inf)) == 255
    assert derive.surface_dice_threshold(np.nextafter(np.sqrt(2) / 2, -np.inf)) == 1


def test_tolerance_validation():
    assert derive.surface_dice_tolerances(2) == (2.0,)
    assert derive.surface_dice_tolerances([2.0, 1.0]) == (2.0, 1.0)
    assert derive.surface_dice_tolerances(np.array([0.0, 8.0])) == (0.0, 8.0)
    for bad in ((), [1, 2, 3, 4, 5], -0.5, float("nan"), 8.000001, [1.0, float("inf")], "x"):
        with pytest.raises(ValueError):
            derive.surface_dice_tolerances(bad)


def test_nsd_nan_and_zero_cases():
    n_surf = np.array([[0, 0], [0, 7], [5, 0], [4, 6]], dtype=np.uint32)
    n_within = np.zeros((4, 2, 2), dtype=np.uint32)
    n_within[3] = [[6, 3], [4, 1]]                       # direction 0 counts pred vertices, 1 true vertices
    got = derive.surface_dice(n_surf, n_within)
    assert got.shape == (4, 2) and got.dtype == np.float64
    assert np.isnan(got[0]).all()
    assert (got[1] == 0).all() and (got[2] == 0).all()
    np.testing.assert_array_equal(got[3], [(6 + 4) / 10, (3 + 1) / 10])
    assert derive.surface_dice(np.zeros((0, 3, 2)), np.zeros((0, 3, 2, 2))).shape == (0, 3, 2)


def _rand_pairs(seed, count):
    rng = np.random.default_rng(seed)
    for _ in range(count):
        h, w = rng.integers(1, 21, size=2)
        a = rng.random((h, w)) < rng.uniform(0.05, 0.95)
        b = rng.random((h, w)) < rng.uniform(0.05, 0.95)
        yield a, b


def test_oracle_brute_force_equals_edt_and_counts_are_monotone():
    from oracle.contours_oracle import directed_sq_distances
    taus = sorted(BOUNDARY_TAUS + (1.5, 2.0, 3.0))
    for a, b in _rand_pairs(11, 40):
        vt, vp = ao.all_vertices(a), ao.all_vertices(b)
        if len(vt) and len(vp):
            np.testing.assert_array_equal(directed_sq_distances(vt, vp), ao.edt_sq_distances(vt, vp, a.shape))
            np.testing.assert_array_equal(directed_sq_distances(vp, vt), ao.edt_sq_distances(vp, vt, a.shape))
        ns, nw = so_.mask_counts(a, b, taus)
        assert ns.tolist() == [len(vt), len(vp)]
        assert (np.diff(nw, axis=1) >= 0).all()
        assert (nw[0] <= ns[1]).all() and (nw[1] <= ns[0]).all()
    same = np.zeros((6, 7), bool)
    same[1:4, 2:6] = True
    ns, nw = so_.mask_counts(same, same, (0.0,))
    assert (nw[:, 0] == ns[::-1]).all() and ns[0] > 0         # identical boundaries: everything within 0


# ---------------------------------------------------------------------------------- C ABI argument checks
@pytest.fixture(scope="module")
def so():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails


def _call(so, *, n=1, h=8, w=8, k=2, thr=(4,), n_thr=None, ptr=FAKE, thr_ptr=True):
    arr = (ctypes.c_uint32 * max(1, len(thr)))(*thr) if thr_ptr else None
    return so.octm_surface_dice_u8(ptr, ptr, n, h, w, k, arr, len(thr) if n_thr is None else n_thr, ptr, ptr, None)


def test_abi_bad_num_classes_and_shape(so):
    assert _call(so, k=99) == -1 and b"num_classes" in so.octm_last_error()
    assert _call(so, k=1) == -1
    assert _call(so, n=-1) == -1
    assert _call(so, h=0) == -1
    assert _call(so, w=9000) == -2


def test_abi_null_pointers(so):
    assert _call(so, ptr=None) == -1 and b"null" in so.octm_last_error()
    assert _call(so, thr_ptr=False) == -1 and b"thresholds_sq" in so.octm_last_error()
    assert so.octm_surface_dice_u8(FAKE, None, 1, 8, 8, 2, (ctypes.c_uint32 * 1)(4), 1, FAKE, FAKE, None) == -1


def test_abi_thresholds(so):
    assert _call(so, thr=(), n_thr=0) == -1 and b"n_thresholds" in so.octm_last_error()
    assert _call(so, thr=(1, 2, 3, 4, 5)) == -1 and b"n_thresholds" in so.octm_last_error()
    assert _call(so, thr=(257,)) == -1 and b"256" in so.octm_last_error()
    assert _call(so, thr=(4, 300)) == -1
    assert _call(so, thr=(16, 4)) == -1 and b"ascending" in so.octm_last_error()


def test_abi_empty_batch_is_a_no_op(so):
    assert _call(so, n=0, ptr=None) == 0
    assert _call(so, n=0, ptr=None, thr=(0, 2, 4, 256)) == 0
    assert _call(so, n=0, ptr=None, thr=(300,)) == -1          # the thresholds are still checked


# ---------------------------------------------------------------------------------- dataset view over ranks
K, H, W, N = 4, 20, 24, 7
TAUS = (1.0, 2.0)


def _fake_result(yt, yp):
    """What a rank's evaluate(surface_dice=TAUS) result holds, with the counts built from the oracle (no GPU here)."""
    ns, nw = so_.label_counts(yt, yp, K, TAUS)
    ints = {"surface_dice_n_surf": ns.astype(np.uint32), "surface_dice_n_within": nw.astype(np.uint32)}
    return types.SimpleNamespace(surface_dice_tolerances=TAUS, integers=lambda: ints)


def _inputs():
    yt, yp = synth.lesion_pair(N, H, W, K, seed=91, single_blob_interior=False)
    yp[0] = yt[0]
    yt[1][yt[1] == 3] = 0                     # class 3 absent from one map of item 1
    yp[1][yp[1] == 3] = 0                     # ... and from both: NSD undefined there
    return yt, yp


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
    yt, yp = _inputs()
    s, e = odist.shard_range(N, rank, world)
    out = odist.surface_dice_totals(_fake_result(yt[s:e], yp[s:e]), world, device="cpu")
    q.put((rank, out["surface_dice_mean"], out["surface_dice_items"], out["tolerances"]))
    torch.distributed.destroy_process_group()


def test_two_rank_surface_dice_totals_equal_a_single_process():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {r: (m, c, t) for r, m, c, t in (q.get(timeout=120) for _ in range(2))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    yt, yp = _inputs()
    single = odist.surface_dice_totals(_fake_result(yt, yp), 1)
    ns, nw = so_.label_counts(yt, yp, K, TAUS)
    nsd = derive.surface_dice(ns, nw)
    assert single["surface_dice_items"][3].tolist() == [N - 1, N - 1]
    np.testing.assert_array_equal(single["surface_dice_items"], (~np.isnan(nsd)).sum(0))
    np.testing.assert_allclose(single["surface_dice_mean"], np.nanmean(nsd, axis=0), rtol=1e-12)
    for r in range(2):
        mean, items, taus = got[r]
        assert taus == TAUS
        np.testing.assert_array_equal(items, single["surface_dice_items"])
        np.testing.assert_allclose(mean, single["surface_dice_mean"], rtol=1e-12)
    with pytest.raises(ValueError, match="surface_dice"):
        odist.surface_dice_totals(types.SimpleNamespace(surface_dice_tolerances=None), 1)
