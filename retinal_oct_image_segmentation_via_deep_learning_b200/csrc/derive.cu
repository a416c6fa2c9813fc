// Float64 epilogue on the device: the reference's scalar expressions evaluated per (item, class)
// from the exact integers of the label pass and the contour kernels, plus the deterministic
// dataset-level reduction that feeds the multi-GPU all-reduce.  sm_100a.
//
// Expression order follows the reference lines cited in derive.py (the host mirror of this file;
// tests/test_gpu_derive.py requires the two to agree bit for bit):
//   Metrics/ConfusionMatrix_based_metrics.py:14-17,30-32,45-47,60-62
//   Metrics/Region_based_metrics.py:13-15,28-30,43-45,58-60
//   Metrics/PixelError_based_metrics.py:14-17,32-35   Metrics/Biomarker_based_metrics.py:18-21,34-38
//   Metrics/Contour_based_metrics.py:22,39,56,68-71   (numpy linear percentile for hd95)
// Multiplications that feed an addition use __dmul_rn/__dadd_rn so nvcc cannot contract them
// into an FMA (numpy rounds after each operation).
#include <cmath>
#include <type_traits>

#include "common.cuh"

namespace octm {

constexpr double kEps = 1e-7;

struct DeriveParams {
    const unsigned long long* counts;   // [n][K][K]
    const long long* thick;             // [n][K] or null
    const long long* bsq;               // [n][K-1] or null
    const long long* babs;              // [n][K-1] or null
    const uint32_t* n_pts;              // [n][K][2] or null (no contour metrics)
    const void* max_sq;                 // [n][K][2]     uint32 (pixel units) or float64 (with a spacing)
    const void* p95_sq;                 // [n][K][2][2]
    const double* sum_dist;             // [n][K][2]
    long long n_items;
    int H, W, K;
    double* cls;                        // [n][K][OCTM_NUM_CLASS_METRICS]
    double* bnd;                        // [n][K-1][3] or null
    double* n_bad;                      // totals slot "n_bad_label_items" (zeroed before the launch) or null
    double sy, wy;                      // with a spacing: the row (axial) spacing and its square
};

template <class SQ>
__device__ __forceinline__ double percentile95(SQ lo_sq, SQ hi_sq, uint32_t m) {
    const double pos = __dmul_rn(static_cast<double>(m - 1), 0.95);     // numpy: (n - 1) * quantile
    const double gamma = pos - floor(pos);
    const double a = sqrt(static_cast<double>(lo_sq) / 4.0), b = sqrt(static_cast<double>(hi_sq) / 4.0);
    const double d = b - a;                                              // numpy _lerp(a, b, t)
    if (gamma >= 0.5) return __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, gamma)));
    return __dadd_rn(a, __dmul_rn(d, gamma));
}

// SPACING: float64 squared contour distances (octm_contour2d_distance_spacing) and the thickness and boundary errors
// scaled by the row spacing: thickness (sum / W) * sy, boundary MSE (sum / W) * wy, MAD (sum / W) * sy.
template <bool SPACING>
__global__ void __launch_bounds__(128) derive_kernel(const DeriveParams p) {
    using SQ = typename std::conditional<SPACING, double, uint32_t>::type;
    const SQ* max_sq = static_cast<const SQ*>(p.max_sq);
    const SQ* p95_sq = static_cast<const SQ*>(p.p95_sq);
    const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int K = p.K;
    if (gid >= p.n_items * K) return;
    const long long item = gid / K;
    const int c = static_cast<int>(gid % K);
    const unsigned long long* cm = p.counts + item * K * K;
    long long row = 0, colsum = 0, total = 0;
    for (int t = 0; t < K; ++t)
        for (int q = 0; q < K; ++q) {
            const long long v = static_cast<long long>(cm[t * K + q]);
            total += v;
            if (t == c) row += v;
            if (q == c) colsum += v;
        }
    // the label pass drops pixels whose label is >= K: such an item's counts do not add up to H * W
    if (c == 0 && p.n_bad != nullptr && total != static_cast<long long>(p.H) * p.W) atomicAdd(p.n_bad, 1.0);
    const long long tp = static_cast<long long>(cm[c * K + c]);
    const long long fn = row - tp, fp = colsum - tp, tn = total - tp - fn - fp;
    const long long st = tp + fn, sp = tp + fp;
    const double n = static_cast<double>(total);
    double* o = p.cls + gid * OCTM_NUM_CLASS_METRICS;
    const double dtp = static_cast<double>(tp), dtn = static_cast<double>(tn);
    o[OCTM_M_ACCURACY] = static_cast<double>(tp + tn) / n;
    o[OCTM_M_SENSITIVITY] = dtp / (static_cast<double>(tp + fn) + kEps);
    o[OCTM_M_CM_PRECISION] = dtp / (static_cast<double>(tp + fp) + kEps);
    o[OCTM_M_SPECIFICITY] = dtn / (static_cast<double>(tn + fp) + kEps);
    o[OCTM_M_DICE] = (2.0 * dtp) / (static_cast<double>(st + sp) + kEps);
    o[OCTM_M_IOU] = dtp / (static_cast<double>(st + sp - tp) + kEps);
    o[OCTM_M_REGION_PRECISION] = dtp / (static_cast<double>(sp) + kEps);
    o[OCTM_M_RECALL] = dtp / (static_cast<double>(st) + kEps);
    const double err = static_cast<double>(fp + fn) / n;
    o[OCTM_M_MSE] = err;
    o[OCTM_M_RMSE] = sqrt(err);
    o[OCTM_M_MAD] = err;
    o[OCTM_M_VASCULARITY] = fabs(static_cast<double>(st) / n - static_cast<double>(sp) / n);
    double thick = p.thick ? static_cast<double>(p.thick[gid]) / static_cast<double>(p.W) : nan("");
    if (SPACING) thick = __dmul_rn(thick, p.sy);
    o[OCTM_M_THICKNESS_DIFF] = thick;
    double hd = nan(""), hd95 = nan(""), assd = nan("");
    if (p.n_pts != nullptr) {
        const uint32_t nt = p.n_pts[gid * 2 + 0], np = p.n_pts[gid * 2 + 1];
        if (nt > 0 && np > 0) {
            const uint32_t m0 = np, m1 = nt;       // query counts: direction 0 = pred vertices, 1 = true vertices
            hd = sqrt(static_cast<double>(max(max_sq[gid * 2], max_sq[gid * 2 + 1])) / 4.0);
            hd95 = fmax(percentile95(p95_sq[gid * 4 + 0], p95_sq[gid * 4 + 1], m0),
                        percentile95(p95_sq[gid * 4 + 2], p95_sq[gid * 4 + 3], m1));
            assd = __dadd_rn(p.sum_dist[gid * 2] / static_cast<double>(m0), p.sum_dist[gid * 2 + 1] / static_cast<double>(m1)) / 2.0;
        }
    }
    o[OCTM_M_HAUSDORFF] = hd;
    o[OCTM_M_HAUSDORFF95] = hd95;
    o[OCTM_M_ASSD] = assd;
    if (p.bnd != nullptr && p.bsq != nullptr && c < K - 1) {
        const long long b = item * (K - 1) + c;
        double mse = static_cast<double>(p.bsq[b]) / static_cast<double>(p.W);
        double mad = static_cast<double>(p.babs[b]) / static_cast<double>(p.W);
        if (SPACING) {
            mse = __dmul_rn(mse, p.wy);
            mad = __dmul_rn(mad, p.sy);
        }
        p.bnd[b * 3 + 0] = mse;
        p.bnd[b * 3 + 1] = sqrt(mse);
        p.bnd[b * 3 + 2] = mad;
    }
}

// Dataset-level partial sums of this rank, one CTA per output element, fixed reduction order
// (thread-strided partials, then a shuffle/shared-memory tree): bit-reproducible run to run.
// Layout (mirrors dist.local_partials): [n_items | cm K*K | thick K | bsq K-1 | babs K-1 |
//   contour_items K | sum hd K | sum hd95 K | sum assd K | n_overflow_items | n_bad_label_items |
//   max hd K | OR of contour flags]
// The first octm_totals_sum_len(K) entries are SUM-reducible across ranks; n_overflow_items counts the items
// with a contour-overflow flag and n_bad_label_items those whose confusion counts do not add up to H * W (the
// label pass drops pixels whose label is >= K), so that every rank of a multi-GPU job takes the same decision
// (retry / raise) from the reduced vector.
struct TotalsParams {
    const unsigned long long* counts;
    const long long* thick;
    const long long* bsq;
    const long long* babs;
    const double* cls;         // [n][K][OCTM_NUM_CLASS_METRICS]
    const uint32_t* flags;     // [n][K] or null
    long long n_items;
    int K;
    double* out;
};

__global__ void __launch_bounds__(256) totals_kernel(const TotalsParams p) {
    __shared__ double s_d[8];
    __shared__ long long s_i[8];
    const int K = p.K, e = blockIdx.x, tid = threadIdx.x;
    const int o_cm = 1, o_th = o_cm + K * K, o_bs = o_th + K, o_ba = o_bs + K - 1, o_nv = o_ba + K - 1;
    const int o_hd = o_nv + K, o_h95 = o_hd + K, o_as = o_h95 + K, o_ov = o_as + K, o_bad = o_ov + 1, o_mx = o_bad + 1,
              o_fl = o_mx + K;
    long long isum = 0;
    double dsum = 0.0, dmax = -1.0;
    bool is_int = true, is_max = false;
    if (e == 0) {
        if (tid == 0) p.out[0] = static_cast<double>(p.n_items);
        return;
    }
    if (e == o_bad) return;          // counted by derive_kernel (which sums every item's counts anyway)
    for (long long i = tid; i < p.n_items; i += 256) {
        if (e < o_th) isum += static_cast<long long>(p.counts[i * K * K + (e - o_cm)]);
        else if (e < o_bs) isum += p.thick ? p.thick[i * K + (e - o_th)] : 0;
        else if (e < o_ba) isum += p.bsq ? p.bsq[i * (K - 1) + (e - o_bs)] : 0;
        else if (e < o_nv) isum += p.babs ? p.babs[i * (K - 1) + (e - o_ba)] : 0;
        else if (e < o_hd) { const double v = p.cls[(i * K + (e - o_nv)) * OCTM_NUM_CLASS_METRICS + OCTM_M_HAUSDORFF]; isum += (v == v) ? 1 : 0; }
        else if (e < o_ov) {
            is_int = false;
            const int which = (e - o_hd) / K, c = (e - o_hd) % K;
            const double v = p.cls[(i * K + c) * OCTM_NUM_CLASS_METRICS + OCTM_M_HAUSDORFF + which];
            if (v == v) dsum += v;
        } else if (e == o_ov) {
            uint32_t f = 0;
            for (int c = 0; c < K; ++c) f |= p.flags ? p.flags[i * K + c] : 0;
            isum += (f & (OCTM_CF_TRUE_OVERFLOW | OCTM_CF_PRED_OVERFLOW)) ? 1 : 0;
        } else if (e < o_fl) {
            is_int = false; is_max = true;
            const double v = p.cls[(i * K + (e - o_mx)) * OCTM_NUM_CLASS_METRICS + OCTM_M_HAUSDORFF];
            if (v == v) dmax = fmax(dmax, v);
        } else {
            for (int c = 0; c < K; ++c) isum |= p.flags ? p.flags[i * K + c] : 0;
        }
    }
    const bool is_or = e == o_fl;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long oi = __shfl_xor_sync(0xffffffffu, isum, o);
        isum = is_or ? (isum | oi) : (isum + oi);
        dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
        dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    }
    if ((tid & 31) == 0) { s_i[tid >> 5] = isum; s_d[tid >> 5] = is_max ? dmax : dsum; }
    __syncthreads();
    if (tid == 0) {
        long long it = 0;
        double dt = is_max ? -1.0 : 0.0;
        for (int w = 0; w < 8; ++w) {
            it = is_or ? (it | s_i[w]) : (it + s_i[w]);
            dt = is_max ? fmax(dt, s_d[w]) : dt + s_d[w];
        }
        p.out[e] = is_int ? static_cast<double>(it) : dt;
    }
}

}  // namespace octm

extern "C" int octm_totals_len(int num_classes) {
    const int K = num_classes;
    return 1 + K * K + K + 2 * (K - 1) + 4 * K + 2 + K + 1;
}

extern "C" int octm_totals_sum_len(int num_classes) {
    const int K = num_classes;
    return 1 + K * K + K + 2 * (K - 1) + 4 * K + 2;
}

static int derive_metrics(const uint64_t* counts, const int64_t* thick_absdiff, const int64_t* bnd_sq, const int64_t* bnd_abs,
                          const uint32_t* n_pts, const void* max_sq, const void* p95_sq, const double* sum_dist,
                          const uint32_t* contour_flags, int64_t n_items, int H, int W, int num_classes,
                          const double* spacing, double* class_metrics, double* boundary_metrics, double* totals,
                          void* stream) {
    if (n_items < 0 || num_classes < 2 || num_classes > OCTM_MAX_CLASSES || W < 1 || H < 1)
        return octm::fail(OCTM_ERR_INVALID, "bad shape");
    if (n_items > 0 && (!counts || !class_metrics)) return octm::fail(OCTM_ERR_INVALID, "counts and class_metrics are required");
    if (n_pts && (!max_sq || !p95_sq || !sum_dist)) return octm::fail(OCTM_ERR_INVALID, "incomplete contour inputs");
    if (boundary_metrics && (!bnd_sq || !bnd_abs)) return octm::fail(OCTM_ERR_INVALID, "boundary sums missing");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    octm::DeriveParams p{reinterpret_cast<const unsigned long long*>(counts), reinterpret_cast<const long long*>(thick_absdiff),
                         reinterpret_cast<const long long*>(bnd_sq), reinterpret_cast<const long long*>(bnd_abs), n_pts, max_sq,
                         p95_sq, sum_dist, n_items, H, W, num_classes, class_metrics, boundary_metrics,
                         totals ? totals + (octm_totals_sum_len(num_classes) - 1) : nullptr,
                         spacing ? spacing[0] : 1.0, spacing ? spacing[0] * spacing[0] : 1.0};
    if (totals != nullptr && cudaMemsetAsync(p.n_bad, 0, sizeof(double), s) != cudaSuccess)
        return octm::fail(OCTM_ERR_LAUNCH, "memset(totals) failed");
    const long long threads = n_items * num_classes;
    if (n_items > 0) {
        const unsigned grid = static_cast<unsigned>((threads + 127) / 128);
        if (spacing) OCTM_TIMED("derive_kernel", s) octm::derive_kernel<true><<<grid, 128, 0, s>>>(p);
        else OCTM_TIMED("derive_kernel", s) octm::derive_kernel<false><<<grid, 128, 0, s>>>(p);
        if (int e = octm::check_launch("derive_kernel")) return e;
    }
    if (totals != nullptr) {       // also for an empty batch: n_items 0, sums 0, maxima -1, flags 0
        octm::TotalsParams t{p.counts, p.thick, p.bsq, p.babs, class_metrics, contour_flags, n_items, num_classes, totals};
        OCTM_TIMED("totals_kernel", s) octm::totals_kernel<<<octm_totals_len(num_classes), 256, 0, s>>>(t);
        if (int e = octm::check_launch("totals_kernel")) return e;
    }
    return OCTM_OK;
}

extern "C" int octm_derive_metrics(const uint64_t* counts, const int64_t* thick_absdiff, const int64_t* bnd_sq,
                                   const int64_t* bnd_abs, const uint32_t* n_pts, const uint32_t* max_sq,
                                   const uint32_t* p95_sq, const double* sum_dist, const uint32_t* contour_flags,
                                   int64_t n_items, int H, int W, int num_classes, double* class_metrics,
                                   double* boundary_metrics, double* totals, void* stream) {
    return derive_metrics(counts, thick_absdiff, bnd_sq, bnd_abs, n_pts, max_sq, p95_sq, sum_dist, contour_flags, n_items,
                          H, W, num_classes, nullptr, class_metrics, boundary_metrics, totals, stream);
}

extern "C" int octm_derive_metrics_spacing(const uint64_t* counts, const int64_t* thick_absdiff, const int64_t* bnd_sq,
                                           const int64_t* bnd_abs, const uint32_t* n_pts, const double* max_sq,
                                           const double* p95_sq, const double* sum_dist, const uint32_t* contour_flags,
                                           int64_t n_items, int H, int W, int num_classes, const double* spacing,
                                           double* class_metrics, double* boundary_metrics, double* totals, void* stream) {
    if (spacing == nullptr) return octm::fail(OCTM_ERR_INVALID, "null pointer: spacing");
    for (int a = 0; a < 2; ++a)
        if (!std::isfinite(spacing[a]) || !(spacing[a] > 0.0) || !std::isnormal(spacing[a] * spacing[a]))
            return octm::fail(OCTM_ERR_INVALID, "spacing[%d] = %g: must be finite and > 0 with a normal square", a, spacing[a]);
    return derive_metrics(counts, thick_absdiff, bnd_sq, bnd_abs, n_pts, max_sq, p95_sq, sum_dist, contour_flags, n_items,
                          H, W, num_classes, spacing, class_metrics, boundary_metrics, totals, stream);
}
