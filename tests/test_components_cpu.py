"""CPU tier of the connected-component metrics: the oracle against an independent flood fill, the NaN/0 rules of
derive.component_metrics, argument validation of evaluate(components=...) and octm_components_u8, and the multi-rank
dataset view."""
import ctypes
import os
import socket
import types
from collections import deque

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from retinal_oct_image_segmentation_via_deep_learning_b200 import derive, synth
from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
import components_oracle as co


def _flood(mask, other, connectivity):
    h, w = mask.shape
    steps = [(-1, 0), (1, 0), (0, -1), (0, 1)]
    if connectivity == 8:
        steps += [(-1, -1), (-1, 1), (1, -1), (1, 1)]
    seen = np.zeros_like(mask, bool)
    n = hits = 0
    for y0 in range(h):
        for x0 in range(w):
            if not mask[y0, x0] or seen[y0, x0]:
                continue
            n += 1
            hit = False
            seen[y0, x0] = True
            todo = deque([(y0, x0)])
            while todo:
                y, x = todo.popleft()
                hit |= bool(other[y, x])
                for dy, dx in steps:
                    v, u = y + dy, x + dx
                    if 0 <= v < h and 0 <= u < w and mask[v, u] and not seen[v, u]:
                        seen[v, u] = True
                        todo.append((v, u))
            hits += hit
    return n, hits


@pytest.mark.parametrize("connectivity", [4, 8])
def test_oracle_equals_flood_fill(connectivity):
    rng = np.random.default_rng(7 + connectivity)
    for it in range(120):
        h, w = (1, 1) if it == 0 else rng.integers(1, 25, size=2)
        k = int(rng.integers(2, 6))
        yt = rng.integers(0, k, size=(1, h, w)).astype(np.uint8)
        yp = yt.copy() if it % 7 == 0 else rng.integers(0, k, size=(1, h, w)).astype(np.uint8)
        nc, nh = co.label_counts(yt, yp, k, connectivity)
        for c in range(k):
            mt, mp = yt[0] == c, yp[0] == c
            assert (nc[0, c, 0], nh[0, c, 0]) == _flood(mt, mp, connectivity)
            assert (nc[0, c, 1], nh[0, c, 1]) == _flood(mp, mt, connectivity)


def test_checkerboard_counts():
    yy, xx = np.mgrid[:5, :7]
    board = ((yy + xx) % 2).astype(np.uint8)[None]
    nc4, _ = co.label_counts(board, board, 2, 4)
    nc8, nh8 = co.label_counts(board, board, 2, 8)
    assert nc4[0, :, 0].tolist() == [18, 17]
    assert nc8[0].tolist() == [[1, 1], [1, 1]] and nh8[0].tolist() == [[1, 1], [1, 1]]


def test_component_metrics_rules():
    n_comp = np.array([[0, 0], [3, 0], [0, 2], [4, 5], [2, 3], [1, 1]], dtype=np.uint32)
    n_hit = np.array([[0, 0], [0, 0], [0, 0], [3, 2], [0, 0], [1, 1]], dtype=np.uint32)
    m = derive.component_metrics(n_comp, n_hit)
    assert set(m) == set(derive.COMPONENT_METRICS)
    for v in m.values():
        assert v.shape == (6,) and v.dtype == np.float64
    np.testing.assert_array_equal(m["component_count_error"], [0, 3, 2, 1, 1, 0])
    r, p, f = m["component_recall"], m["component_precision"], m["component_f1"]
    assert np.isnan(r[0]) and np.isnan(p[0]) and np.isnan(f[0])            # no component in either map
    assert r[1] == 0 and np.isnan(p[1]) and f[1] == 0                         # nothing predicted
    assert np.isnan(r[2]) and p[2] == 0 and f[2] == 0                         # nothing true
    assert r[3] == 3 / 4 and p[3] == 2 / 5 and f[3] == 2 * (2 / 5) * (3 / 4) / (2 / 5 + 3 / 4)
    assert r[4] == 0 and p[4] == 0 and f[4] == 0                              # P + R == 0
    assert r[5] == p[5] == f[5] == 1.0
    empty = derive.component_metrics(np.zeros((0, 4, 2), np.uint32), np.zeros((0, 4, 2), np.uint32))
    assert all(v.shape == (0, 4) for v in empty.values())


def test_components_argument_validation():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    for ok in (4, 8, np.int64(8)):
        assert suite._connectivity(ok) in (4, 8)
    t = torch.zeros((1, 4, 4), dtype=torch.uint8)
    for bad in (0, 6, "4", True, 4.5, (4,), 16):
        with pytest.raises(ValueError, match="components"):
            suite._connectivity(bad)
        with pytest.raises(ValueError, match="components"):
            suite.evaluate(t, t, 2, components=bad)           # rejected before anything touches the device
        with pytest.raises(ValueError, match="components"):
            suite.components(t, t, 2, bad)


# ---------------------------------------------------------------------------------- C ABI argument checks
@pytest.fixture(scope="module")
def so():
    from retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build import build_library
    build_library()
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib
    return _lib.load()


FAKE = ctypes.c_void_p(256)      # a non-null device address; never dereferenced when validation fails


def _call(so, *, n=1, h=8, w=8, k=2, conn=4, ptr=FAKE):
    return so.octm_components_u8(ptr, ptr, n, h, w, k, conn, ptr, ptr, None)


def test_abi_connectivity(so):
    for bad in (0, 2, 6, -4, 9):
        assert _call(so, conn=bad) == -1 and b"connectivity" in so.octm_last_error()
    assert _call(so, n=0, ptr=None, conn=6) == -1                 # checked on an empty batch too


def test_abi_bad_num_classes_and_shape(so):
    assert _call(so, k=17) == -1 and b"num_classes" in so.octm_last_error()
    assert _call(so, k=1) == -1
    assert _call(so, n=-1) == -1
    assert _call(so, h=0) == -1
    assert _call(so, w=0) == -1
    assert _call(so, w=9000) == -2


def test_abi_null_pointers(so):
    assert _call(so, ptr=None) == -1 and b"null" in so.octm_last_error()
    assert so.octm_components_u8(FAKE, None, 1, 8, 8, 2, 8, FAKE, FAKE, None) == -1
    assert so.octm_components_u8(FAKE, FAKE, 1, 8, 8, 2, 8, FAKE, None, None) == -1


def test_abi_empty_batch_is_a_no_op(so):
    assert _call(so, n=0, ptr=None) == 0
    assert _call(so, n=0, ptr=None, conn=8, k=16) == 0


# ---------------------------------------------------------------------------------- dataset view over ranks
K, H, W, N = 4, 20, 24, 7
CONN = 8


def _fake_result(yt, yp):
    """What a rank's evaluate(components=CONN) result holds, with the counts built from the oracle (no GPU here)."""
    nc, nh = co.label_counts(yt, yp, K, CONN)
    ints = {"component_count": nc.astype(np.uint32), "component_hits": nh.astype(np.uint32)}
    return types.SimpleNamespace(component_connectivity=CONN, integers=lambda: ints)


def _inputs():
    yt, yp = synth.lesion_pair(N, H, W, K, seed=93, single_blob_interior=False)
    yp[0] = yt[0]
    yt[1][yt[1] == 3] = 0
    yp[1][yp[1] == 3] = 0
    return yt, yp


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
    yt, yp = _inputs()
    s, e = odist.shard_range(N, rank, world)
    q.put((rank, odist.component_totals(_fake_result(yt[s:e], yp[s:e]), world, device="cpu")))
    torch.distributed.destroy_process_group()


def test_two_rank_component_totals_equal_a_single_process():
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
        assert p.exitcode == 0
    yt, yp = _inputs()
    single = odist.component_totals(_fake_result(yt, yp), 1)
    nc, nh = co.label_counts(yt, yp, K, CONN)
    np.testing.assert_array_equal(single["component_count"], nc.sum(0))
    np.testing.assert_array_equal(single["component_hits"], nh.sum(0))
    assert single["items"] == N and single["connectivity"] == CONN
    pooled = derive.component_metrics(nc.sum(0), nh.sum(0))
    for key in ("component_recall", "component_precision", "component_f1"):
        np.testing.assert_array_equal(single[key], pooled[key], err_msg=key)
    np.testing.assert_array_equal(single["component_count_error"], np.abs(nc[..., 0] - nc[..., 1]).mean(0))
    for r in range(2):
        for key, v in single.items():
            np.testing.assert_array_equal(got[r][key], v, err_msg=key)
    with pytest.raises(ValueError, match="components"):
        odist.component_totals(types.SimpleNamespace(component_connectivity=None), 1)
