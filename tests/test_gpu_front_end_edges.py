"""GPU parity of the front end and helper kernels at their routes, grid strides and edges: the argmax
(``argmax_planes_kernel``, ``argmax_generic_kernel``), ROC AUC (``auc_kernel``), boundary rows -> label maps
(``rasterise_kernel``) and the soft boundary errors and topology violations (``boundary_error_float_kernel``,
``topology_kernel``).

Every case asserts the route it is meant to reach: the argmax kernel by name from ``_lib.kernel_profile()``, the other
kernels by the input property that forces the route (width modulo 4, key width, rows or pairs above the fixed grid,
items above the SM count).  Integer outputs are compared bit for bit; float outputs against a plain float64 reference:
the exact rank-sum quotient for AUC (and scikit-learn), ``math.fsum`` for the boundary sums."""
import math

import numpy as np
import pytest
import torch
from sklearn.metrics import roc_auc_score

from oracle import labelmap_oracle as lo
from oracle import metrics_oracle as mo
from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite, synth

pytestmark = pytest.mark.gpu

ARGMAX_THREADS = 256                                   # both argmax kernels
ARGMAX_PLANES_CTAS_PER_SM, ARGMAX_GENERIC_CTAS_PER_SM = 8, 16
VPT = {torch.float32: 8, torch.float16: 16, torch.bfloat16: 16}      # scores per 32-byte vector of the planes kernel
AUC_THREADS = 1024                                     # auc_kernel: one CTA per item, a contiguous chunk per thread
RASTER_THREADS, RASTER_CTAS_PER_SM = 128, 16           # rasterise_kernel: a strip is 128 * V columns
ROW_GRID = 148 * 16                                    # boundary_error_float_kernel / topology_kernel: grid cap
U = 2.0**-53                                           # float64 unit roundoff
INT_MIN, INT_MAX = -(2**31), 2**31 - 1
SCORE_DTYPES = [torch.float32, torch.float16, torch.bfloat16]
AUC_DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]


@pytest.fixture(scope="module")
def sms(cuda):
    return torch.cuda.get_device_properties(cuda).multi_processor_count


def _tiny(dtype):
    """The smallest positive subnormal of ``dtype``."""
    fi = torch.finfo(dtype)
    return fi.smallest_normal * fi.eps


# ------------------------------------------------------------------------------------------------------------ argmax
def _argmax(scores, **kw):
    """labels_from_scores -> (labels as numpy, name of the one kernel it launched)."""
    with _lib.kernel_profile() as prof:
        got = suite.labels_from_scores(scores, **kw)
        torch.cuda.synchronize()
    assert len(prof.kernels) == 1, prof.kernels
    return got.cpu().numpy(), next(iter(prof.kernels))


def _argmax_ref(x, axis=1):
    # numpy argmax of the float32 upcast: the first maximal class, a NaN counts as maximal
    return np.argmax(x.float().numpy(), axis=axis).astype(np.uint8)


def _quarter_scores(shape, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    return ((torch.randn(shape, generator=g) * 4).round() / 4).to(dtype)      # many exact ties


def _special_scores(dtype):
    """[1, 5, 16, 16] scores whose first pixels hold the special patterns; ``want`` the expected class of each."""
    x = _quarter_scores((1, 5, 16, 16), torch.float64, 11) - 10.0
    inf, nan, tiny = math.inf, math.nan, _tiny(dtype)
    fmax = torch.finfo(dtype).max
    patterns = [
        ([nan, 0, 0, 0, 0], 0),                        # NaN in class 0
        ([0, 1, nan, 1, nan], 2),                      # NaN in two classes: the first
        ([-inf] * 5, 0),                               # every class -inf
        ([-inf, nan, -inf, -inf, -inf], 1),            # -inf followed by NaN
        ([-1, -0.0, -1, 0.0, -1], 1),                  # -0.0 tied with +0.0: the first
        ([0.0, -1, -1, -1, -0.0], 0),
        ([0, 0, 0, tiny, 0], 3),                       # a subnormal above zero
        ([-tiny, -0.0, 0, -tiny, 0], 1),               # below zero
        ([0, tiny, 0, 0, 2 * tiny], 4),                # two subnormals
        ([0, inf, nan, inf, 0], 2),                    # NaN after +inf
        ([nan] * 5, 0),
        ([-fmax, fmax, fmax, inf, fmax], 3),
    ]
    want = []
    for p, (vals, cls) in enumerate(patterns):
        x[0, :, p // 16, p % 16] = torch.tensor(vals, dtype=torch.float64)
        want.append(cls)
    return x.to(dtype), want


@pytest.mark.parametrize("dtype", SCORE_DTYPES)
def test_argmax_special_values_on_both_routes(cuda, dtype):
    x, want = _special_scores(dtype)
    ref = _argmax_ref(x)
    assert ref.reshape(-1)[:len(want)].tolist() == want          # the patterns mean what they say under numpy
    got, kern = _argmax(x.to(cuda))
    assert kern == "argmax_planes_kernel"
    np.testing.assert_array_equal(got, ref)
    got, kern = _argmax(x.permute(0, 2, 3, 1).contiguous().to(cuda), channels_last=True)
    assert kern == "argmax_generic_kernel"
    np.testing.assert_array_equal(got, ref)


@pytest.mark.parametrize("dtype", SCORE_DTYPES)
def test_argmax_generic_route_by_misalignment(cuda, dtype):
    """Scores whose P is a multiple of VPT take the planes route only when they start on 32 bytes and ``out=`` on 16."""
    x = _quarter_scores((2, 5, 16, 32), dtype, 12)
    assert (16 * 32) % VPT[dtype] == 0
    ref = _argmax_ref(x)
    got, kern = _argmax(x.to(cuda))
    assert kern == "argmax_planes_kernel"
    np.testing.assert_array_equal(got, ref)
    shift = 4 // x.element_size()
    buf = torch.empty(x.numel() + shift, dtype=dtype, device=cuda)
    s = buf[shift:].view(x.shape)
    s.copy_(x.to(cuda))
    assert s.is_contiguous() and s.data_ptr() % 32 == 4
    got, kern = _argmax(s)
    assert kern == "argmax_generic_kernel"
    np.testing.assert_array_equal(got, ref)
    ob = torch.empty(2 * 16 * 32 + 1, dtype=torch.uint8, device=cuda)
    out = ob[1:].view(2, 16, 32)
    assert out.data_ptr() % 16 == 1
    got, kern = _argmax(x.to(cuda), out=out)
    assert kern == "argmax_generic_kernel"
    np.testing.assert_array_equal(got, ref)


@pytest.mark.parametrize("n,dtype", [(10, torch.float32), (20, torch.float16)])
def test_argmax_planes_grid_stride(cuda, sms, n, dtype):
    x = _quarter_scores((n, 5, 496, 512), dtype, n)
    vectors = n * 496 * 512 // VPT[dtype]
    assert vectors > sms * ARGMAX_PLANES_CTAS_PER_SM * ARGMAX_THREADS
    got, kern = _argmax(x.to(cuda))
    assert kern == "argmax_planes_kernel"
    np.testing.assert_array_equal(got, _argmax_ref(x))


def test_argmax_generic_grid_stride_and_evaluate_scores(cuda, sms):
    """Channels-last scores of 3 x 496 x 512 pixels, more than the generic kernel's grid holds; ``evaluate_scores``
    on them gives the integers ``evaluate`` gives on numpy's argmax."""
    n, k, h, w = 3, 6, 496, 512
    assert n * h * w > sms * ARGMAX_GENERIC_CTAS_PER_SM * ARGMAX_THREADS
    yt, yp = synth.layered_pair(n, h, w, k, seed=33, noise=0.01)
    x = _quarter_scores((n, h, w, k), torch.float32, 13)
    x.scatter_add_(3, torch.from_numpy(yp).long()[..., None], torch.full((n, h, w, 1), 5.0))   # mostly yp
    ref = _argmax_ref(x, axis=3)
    assert 0 < np.count_nonzero(ref != yp) < ref.size // 100
    got, kern = _argmax(x.to(cuda), channels_last=True)
    assert kern == "argmax_generic_kernel"
    np.testing.assert_array_equal(got, ref)
    t = torch.from_numpy(yt).to(cuda)
    a = suite.evaluate(t, torch.from_numpy(ref).to(cuda), k).integers()
    with _lib.kernel_profile() as prof:
        b = suite.evaluate_scores(t, x.to(cuda), channels_last=True).integers()
    assert "argmax_generic_kernel" in prof.kernels
    assert a.keys() == b.keys()
    for key in a:
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)


# --------------------------------------------------------------------------------------------------------------- AUC
def _auc(m, s, cuda, **kw):
    """auc_scores of numpy labels ``m`` [N, P] and CPU scores ``s`` [N, P] -> float64 numpy [N]."""
    return suite.auc_scores(torch.from_numpy(np.ascontiguousarray(m)).to(cuda), s.to(cuda), **kw).cpu().numpy()


def _check_auc(got, m, s, sklearn=True):
    """``got`` equals the exact rank-sum quotient bit for bit, and scikit-learn within 1e-12 relative."""
    s64 = s.to(torch.float64).numpy()
    for i in range(len(got)):
        u2, npos, nneg = mo.auc_rank_sum(m[i], s64[i])
        assert npos and nneg, i
        assert got[i] == u2 / (2.0 * npos * nneg), (i, got[i], u2, npos, nneg)
        if sklearn:
            with np.errstate(over="ignore", invalid="ignore"):              # scores of +-float64 max
                sk = roc_auc_score(m[i], s64[i])
            np.testing.assert_allclose(got[i], sk, rtol=1e-12, atol=0, err_msg=str(i))


def _both_classes(rng, n, p, frac=0.4):
    m = (rng.random((n, p)) < frac).astype(np.uint8)
    m[:, 0], m[:, -1] = 0, 1
    return m


@pytest.mark.parametrize("dtype", AUC_DTYPES)
def test_auc_item_sizes_and_key_widths(cuda, dtype):
    """Items below, at and above a warp (32) and a CTA (1024 threads); float64 sorts 8-byte keys in 8 radix passes,
    the other types 4-byte keys in 4."""
    rng = np.random.default_rng(21)
    for p in (1, 2, 31, 33, 1023, 1025):
        s = torch.from_numpy(np.round(rng.normal(size=(4, p)), 1)).to(dtype)
        if p == 1:
            m = (np.arange(4) % 2).astype(np.uint8)[:, None]
            assert np.isnan(_auc(m, s, cuda)).all()                  # one element: one class
            continue
        m = _both_classes(rng, 4, p)
        _check_auc(_auc(m, s, cuda), m, s)


def test_auc_one_item_of_four_million_elements(cuda):
    rng = np.random.default_rng(22)
    p = 2**22 + 3
    m = (rng.random((1, p)) < 0.3).astype(np.uint8)
    s = (rng.integers(0, 3000, size=(1, p)) + 900 * m.astype(np.int64)) / 16                # heavy ties
    s = torch.from_numpy(s.astype(np.float32))
    _check_auc(_auc(m, s, cuda), m, s, sklearn=False)


def _byte_pattern_scores(rng, shape, nbytes, vary, top):
    """Scores whose key bytes in ``vary`` (0 = least significant) take a few random values and every other byte one
    value: the radix passes of the other bytes find every key on one digit and move nothing."""
    bits = np.zeros(shape, dtype=np.uint64)
    for j in range(nbytes):
        if j == nbytes - 1:
            byte = rng.choice(top, size=shape).astype(np.uint64) if j in vary else np.full(shape, top[0], np.uint64)
        else:
            byte = rng.integers(0, 4, size=shape).astype(np.uint64) if j in vary else np.full(shape, 0x5A, np.uint64)
        bits |= byte << np.uint64(8 * j)
    return bits.astype(np.uint32).view(np.float32) if nbytes == 4 else bits.view(np.float64)


@pytest.mark.parametrize("dtype,vary", [
    (torch.float32, {0, 2}), (torch.float32, {1, 3}), (torch.float32, {0}), (torch.float32, {2}),
    (torch.float64, {0, 2, 4, 6}), (torch.float64, {1, 3, 5, 7}), (torch.float64, {5}), (torch.float64, {0, 7})])
def test_auc_trivial_radix_passes_between_moving_ones(cuda, dtype, vary):
    nbytes = 4 if dtype == torch.float32 else 8
    top = [0x3F, 0x3E] if nbytes == 4 else [0x3F, 0x40]              # one sign: the fixed bytes stay fixed in the keys
    rng = np.random.default_rng(len(vary) * 10 + min(vary))
    s = torch.from_numpy(_byte_pattern_scores(rng, (3, 5000), nbytes, vary, top))
    assert torch.isfinite(s).all()
    m = _both_classes(rng, 3, 5000)
    _check_auc(_auc(m, s, cuda), m, s)


def _chunk_runs(n):
    """Tie runs [a, b] of the sorted sequence placed on the kernel's chunk edges for an item of n elements."""
    tchunk = -(-n // AUC_THREADS)                                    # sweep: a contiguous chunk per thread
    tb = lambda t: min(n, t * tchunk)
    te = lambda t: min(n, tb(t) + tchunk)
    wsweep = 32 * tchunk                                             # a warp's part of the sweep
    wsort = ((-(-n // 32)) + 31) & ~31                               # radix sort: a chunk per warp
    last_t = (n - 1) // tchunk
    return [(0, tchunk), (tb(5), te(5) - 1), (tb(10), te(12) - 1), (te(20) - 1, tb(22)), (tb(25) + 1, te(25) - 2),
            (wsweep - 3, 2 * wsweep + 2), (3 * wsweep, 4 * wsweep - 1), (5 * wsweep - 1, 5 * wsweep),
            (wsort - 2, wsort + 2), (tb(last_t - 40), te(last_t - 38) - 1), (tb(last_t - 3), n - 1)]


@pytest.mark.parametrize("n", [8168, 37893])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_auc_tie_runs_on_chunk_edges(cuda, n, dtype):
    """Constant-score blocks that start or end exactly on a thread's chunk (``tb``, ``te - 1``), span whole thread
    chunks, and cross or fill a warp's part of the sweep; the carries between chunks must join them."""
    runs = _chunk_runs(n)
    assert max(b for _, b in runs) == n - 1 and all(a < b for a, b in runs)
    v = np.arange(n, dtype=np.float64)
    for a, b in runs:
        v[a:b + 1] = v[a]
    rng = np.random.default_rng(n)
    m = (rng.random((2, n)) < 0.5).astype(np.uint8)
    m[:, :2], m[:, -2:] = 0, 1
    perm = rng.permutation(n)
    s = torch.from_numpy(np.stack([v, v[perm]])).to(dtype)
    m[1] = m[1][perm]
    _check_auc(_auc(m, s, cuda), m, s)


@pytest.mark.parametrize("dtype", AUC_DTYPES)
def test_auc_signed_zero_subnormals_and_extremes(cuda, dtype):
    fi, tiny = torch.finfo(dtype), _tiny(dtype)
    vals = np.array([-0.0, 0.0, tiny, -tiny, 2 * tiny, fi.smallest_normal, -fi.smallest_normal, fi.max, -fi.max, 1.0])
    rng = np.random.default_rng(23)
    m = _both_classes(rng, 2, 3000, 0.5)
    s = torch.from_numpy(rng.choice(vals, size=(2, 3000))).to(dtype)
    s[1] = torch.where(torch.from_numpy(m[1]).bool(), -0.0, 0.0).to(dtype)   # positives at -0.0, negatives at +0.0
    assert torch.signbit(s).any() and (s.to(torch.float64).abs() == tiny).any()
    got = _auc(m, s, cuda)
    _check_auc(got, m, s)
    assert got[1] == 0.5                                             # -0.0 == +0.0: one tie


def test_auc_label_values_and_refusals(cuda):
    rng = np.random.default_rng(24)
    m01 = _both_classes(rng, 1, 2000)
    s = torch.from_numpy(np.round(rng.normal(size=(1, 2000)), 1).astype(np.float32))
    ref = _auc(m01, s, cuda)
    _check_auc(ref, m01, s)
    for lo_, hi in ((0, 255), (3, 7)):
        assert _auc(np.where(m01 == 1, hi, lo_).astype(np.uint8), s, cuda)[0] == ref[0], (lo_, hi)
    got = suite.auc_scores(torch.from_numpy(m01.astype(bool)).to(cuda), s.to(cuda)).cpu().numpy()
    assert got[0] == ref[0]
    third = np.repeat(m01, 3, axis=0)
    third[0, 17], third[1, 17], third[2, 17] = 2, 255, 5
    third[2] = np.where(third[2] == 1, 7, np.where(third[2] == 0, 3, third[2]))
    assert (_auc(third, s.repeat(3, 1), cuda) == 0.0).all()          # a third label value
    bad = s.repeat(3, 1)
    bad[0, 5], bad[1, 6], bad[2, 7] = math.nan, math.inf, -math.inf
    for dtype in AUC_DTYPES:
        assert (_auc(np.repeat(m01, 3, axis=0), bad.to(dtype), cuda) == 0.0).all(), dtype    # NaN / inf scores
    single = np.stack([np.zeros(2000, np.uint8), np.ones(2000, np.uint8), np.full(2000, 7, np.uint8)])
    assert np.isnan(_auc(single, s.repeat(3, 1), cuda)).all()
    assert (_auc(single, s.repeat(3, 1), cuda, single_class_value=0.0) == 0.0).all()


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_auc_early_exit_and_normal_items_share_a_cta(cuda, sms, dtype):
    """With more items than SMs, CTA i runs items i, i + sms, ...: an early-exit item (single class, third label,
    NaN or inf score) and a normal one meet on the same CTA, in both orders."""
    n, p = 2 * sms + 8, 1500
    assert n > sms
    rng = np.random.default_rng(25)
    m = _both_classes(rng, n, p)
    s = torch.from_numpy(np.round(rng.normal(size=(n, p)), 1)).to(dtype)
    want = np.full(n, np.nan)
    for j in range(sms):
        i = j if j % 2 == 0 else j + sms                             # the early-exit item of CTA j
        kind = (j // 2) % 4
        if kind == 0:
            m[i] = 1                                                 # single class -> NaN
        elif kind == 1:
            m[i, 3], want[i] = 2, 0.0                                # third label -> 0.0
        elif kind == 2:
            s[i, 4], want[i] = math.nan, 0.0
        else:
            s[i, p - 1], want[i] = math.inf, 0.0
    got = _auc(m, s, cuda)
    early = np.zeros(n, bool)
    early[[j if j % 2 == 0 else j + sms for j in range(sms)]] = True
    np.testing.assert_array_equal(got[early], want[early])          # NaN == NaN here
    normal = np.flatnonzero(~early)
    _check_auc(got[normal], m[normal], s[torch.from_numpy(normal)], sklearn=False)


# --------------------------------------------------------------------------------------------------------- rasterise
def _raster_check(b, h, cuda):
    """labels_from_boundaries of the CPU tensor ``b`` against the oracle on the caller's own dtype, bit for bit."""
    got = suite.labels_from_boundaries(b.to(cuda), h).cpu().numpy()
    np.testing.assert_array_equal(got, lo.labels_from_boundaries(b.numpy(), h))
    return got


def _edge_rows(rng, edges, n, w, dtype):
    """[n, 15, w] rows drawn from ``edges``; column 0 holds 15 equal thresholds and each later column up to len(edges)
    one edge value in every boundary."""
    e = np.array(edges, dtype=dtype)
    b = rng.choice(e, size=(n, 15, w))
    b[:, :, 0] = 5
    for c in range(1, min(w, len(e) + 1)):
        b[:, :, c] = e[c - 1]
    return torch.from_numpy(b)


H = 130
INT_EDGES = [-1, 0, 5, H - 1, H, 100, 101, INT_MIN, INT_MAX, INT_MIN + 1, INT_MAX - 1]
F32_EDGES = [math.inf, -math.inf, 3e9, -3e9, -0.0, 0.0, 1e-45, 5, 3 + 2**-20, 15 + 2**-20, 7 - 2**-20, math.nan,
             H - 1, H - 0.5, 100.5, -1.0, 2147483000.0, -2147483000.0]
F64_EDGES = F32_EDGES + [100.0000001, 99.9999999, 1e-50, -1e-50, 4097 + 2**-20, 100 + 2**-20, 2**31 - 0.5, 2.0**31,
                         -(2.0**31) - 10, 1e300, -1e300]
I64_EDGES = INT_EDGES + [2**32 + 5, 2**32 + 100, -(2**31) - 10, 2**31, -(2**32) + 101, 2**63 - 1, -(2**63)]


@pytest.mark.parametrize("w,v", [(40, 4), (41, 1)])
@pytest.mark.parametrize("dtype", [np.int32, np.float32, np.float64, np.int64])
def test_rasterise_threshold_edges(cuda, w, v, dtype):
    """INT_MIN / INT_MAX, -1, 0, H - 1, H; +-inf, +-3e9, -0.0, 1e-45, k + 2**-20, NaN; and 15 equal thresholds in a
    column, on the V = 4 (w % 4 == 0) and V = 1 routes.  float64 and int64 rows are compared on their own values: a
    float32 / int32 narrowing moves 100.0000001 to row 100, 1e-50 to row 0, 2**32 + 5 to row 5 and -2**31 - 10 to never."""
    edges = {np.int32: INT_EDGES, np.float32: F32_EDGES, np.float64: F64_EDGES, np.int64: I64_EDGES}[dtype]
    rng = np.random.default_rng(w)
    assert (w % 4 == 0) == (v == 4) and w > len(edges)
    b = _edge_rows(rng, edges, 3, w, dtype)
    _raster_check(b, H, cuda)


@pytest.mark.parametrize("n,w,v", [(2500, 512, 4), (1000, 301, 1)])
def test_rasterise_grid_stride(cuda, sms, n, w, v):
    h, kb = 8, 3
    assert (w % 4 == 0) == (v == 4)
    jobs = n * -(-w // (RASTER_THREADS * v))
    assert jobs > sms * RASTER_CTAS_PER_SM
    rng = np.random.default_rng(n)
    _raster_check(torch.from_numpy(rng.integers(-1, h + 1, size=(n, kb, w)).astype(np.int32)), h, cuda)


# ------------------------------------------------------------------------------------- soft boundary errors, topology
def _fsum_rows(t):
    return np.array([math.fsum(r.tolist()) for r in t])


def _within_rounding(got, ref, w):
    """|got - ref| <= (W + 1) u ref: W nonnegative float64 terms summed in any order, against the correctly rounded
    sum of the same terms."""
    assert np.all(np.abs(got - ref) <= (w + 1) * U * ref), np.max(np.abs(got - ref) / np.maximum(ref, 1e-300))


def _boundary_sums(a, b, cuda):
    sq, ab = suite.boundary_error(a.to(cuda), b.to(cuda))
    return sq.cpu().numpy().reshape(-1), ab.cpu().numpy().reshape(-1)


def _dyadic(rng, shape, dtype):
    """Multiples of 1/8 in [0, 64): every partial sum of their squared differences is exact in float64."""
    return torch.from_numpy(rng.integers(0, 512, size=shape) / 8.0).to(dtype)


@pytest.mark.parametrize("n,kb,w", [(300, 9, 1024), (5, 3, 1), (4, 5, 129), (1, 1, 10**6)])
def test_boundary_error_sums(cuda, n, kb, w):
    """Rows above the fixed grid of 2368 CTAs, W = 1, W = 129 and one row of 10**6 positions: float64 rows against
    ``math.fsum`` of the float64 terms within the rounding bound, dyadic rows (float32, and float16 truth against
    float32 prediction) bit for bit."""
    if n == 300:
        assert n * kb > ROW_GRID
    rng = np.random.default_rng(n * kb + w)
    a = torch.from_numpy(rng.normal(100, 30, (n, kb, w)))
    b = a + torch.from_numpy(rng.normal(0, 2, (n, kb, w)))
    d = (a - b).numpy().reshape(n * kb, w)
    sq, ab = _boundary_sums(a, b, cuda)
    _within_rounding(sq, _fsum_rows(d * d), w)
    _within_rounding(ab, _fsum_rows(np.abs(d)), w)
    for ta, tb in ((torch.float32, torch.float32), (torch.float16, torch.float32)):
        a, b = _dyadic(rng, (n, kb, w), ta), _dyadic(rng, (n, kb, w), tb)
        d = (a.to(torch.float64) - b.to(torch.float64)).numpy().reshape(n * kb, w)
        sq, ab = _boundary_sums(a, b, cuda)
        np.testing.assert_array_equal(sq, _fsum_rows(d * d))
        np.testing.assert_array_equal(ab, _fsum_rows(np.abs(d)))


def _topology_ref(pos):
    """relu(pos[k] - pos[k+1]) summed (fsum) and counted per pair, skipping NaN differences."""
    d = pos[:, :-1] - pos[:, 1:]
    with np.errstate(invalid="ignore"):
        hit = d > 0
    flat_d, flat_hit = d.reshape(-1, d.shape[-1]), hit.reshape(-1, d.shape[-1])
    return np.array([math.fsum(r[h].tolist()) for r, h in zip(flat_d, flat_hit)]), flat_hit.sum(-1)


@pytest.mark.parametrize("n,kb,w", [(300, 11, 1024), (3, 2, 1), (2, 4, 129), (1, 2, 10**6)])
def test_topology_violations_sums_and_counts(cuda, n, kb, w):
    """Pairs above the fixed grid of 2368 CTAs (the per-pair count must restart on every pair a CTA takes), W = 1,
    W = 129 and one pair of 10**6 columns."""
    if n == 300:
        assert n * (kb - 1) > ROW_GRID
    rng = np.random.default_rng(n * kb + w + 1)
    pos = np.cumsum(rng.uniform(0, 4, size=(n, kb, w)), axis=1) + rng.normal(0, 2.0, (n, kb, w))
    sv, nv = suite.topology_violations(torch.from_numpy(pos).to(cuda))
    ref_s, ref_n = _topology_ref(pos)
    np.testing.assert_array_equal(nv.cpu().numpy().reshape(-1), ref_n)
    _within_rounding(sv.cpu().numpy().reshape(-1), ref_s, w)
    pos = _dyadic(rng, (n, kb, w), torch.float32)
    sv, nv = suite.topology_violations(pos.to(cuda))
    ref_s, ref_n = _topology_ref(pos.to(torch.float64).numpy())
    np.testing.assert_array_equal(nv.cpu().numpy().reshape(-1), ref_n)
    np.testing.assert_array_equal(sv.cpu().numpy().reshape(-1), ref_s)


def test_nan_and_inf_positions(cuda):
    """A NaN position makes its row's sums NaN and an infinite one inf (NaN for inf - inf), as numpy's mean does.
    ``topology_violations`` skips a column whose difference is NaN in both the sum and the count (NaN = boundary
    absent), where the reference's relu would propagate the NaN; +inf above a finite position is one violation of inf."""
    rng = np.random.default_rng(26)
    a, b = _dyadic(rng, (1, 5, 64), torch.float32), _dyadic(rng, (1, 5, 64), torch.float32)
    a[0, 0, 5] = math.nan
    b[0, 1, 7] = math.inf
    a[0, 2, 9], b[0, 2, 9] = math.inf, math.inf
    b[0, 3, 0] = -math.inf
    sq, ab = _boundary_sums(a, b, cuda)
    a64, b64 = a.to(torch.float64).numpy()[0], b.to(torch.float64).numpy()[0]
    with np.errstate(invalid="ignore"):
        ref_mse = np.mean((a64 - b64) ** 2, axis=-1)
        ref_mad = np.mean(np.abs(a64 - b64), axis=-1)
    np.testing.assert_array_equal(sq / 64, ref_mse)
    np.testing.assert_array_equal(ab / 64, ref_mad)
    assert np.isnan(sq[[0, 2]]).all() and np.isinf(sq[[1, 3]]).all() and np.isfinite(sq[4])

    pos = _dyadic(rng, (1, 4, 64), torch.float32)
    pos[0, 1, 3] = math.nan
    pos[0, 2, 9], pos[0, 3, 9] = math.inf, 1.0
    sv, nv = suite.topology_violations(pos.to(cuda))
    p64 = pos.to(torch.float64).numpy()
    ref_s, ref_n = _topology_ref(p64)
    np.testing.assert_array_equal(nv.cpu().numpy().reshape(-1), ref_n)
    np.testing.assert_array_equal(sv.cpu().numpy().reshape(-1), ref_s)
    assert np.isinf(ref_s[2]) and np.isfinite(ref_s[:2]).all()
    with np.errstate(invalid="ignore"):
        assert np.isnan(np.maximum(p64[0, :-1] - p64[0, 1:], 0.0)[:2].sum(-1)).all()     # the reference's relu
