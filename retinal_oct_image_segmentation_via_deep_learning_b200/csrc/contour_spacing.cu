// Contour distances with a physical pixel spacing (sy, sx) -- sm_100a.
//
// Same vertex lists as octm_contour2d_distance (packed y2 << 16 | x2 on the doubled lattice, from
// octm_contour2d_trace_u8 or octm_contour2d_all_vertices_u8), same units and directions (unit = (item, class, dir);
// direction 0: pred vertices -> true set, 1: true -> pred).  A vertex pair at lattice offset (a, b) is
//     q = fl(fl(wy * a^2) + fl(wx * b^2)),   wy = sy * sy, wx = sx * sx   (float64, in that order),
// a query's d2 is the minimum of q over the source set, and its distance sqrt(d2 / 4.0).  At (1, 1) q is the integer D2
// of the pixel path, exactly.
//
//   distance_spacing_kernel  one CTA per unit (grid-strided).  The unit's source vertices are counting-sorted by column
//                            into shared memory (row only, 2 B each; col[c] .. col[c + 1] is column c), in tiles of
//                            kSpTile vertices when a list is longer.  One thread per query searches outward by column,
//                            b = 0, 1, 2, ..: column qx +- b can hold a nearer vertex only while fl(wx * b^2) <= best
//                            (q >= fl(wx * b^2): the other term is >= 0 and rounding is monotone), so stopping there is
//                            exact.  The minima go to shared memory (or to d2 when stored) and give, with no histogram:
//                            the max, sum sqrt(d2 / 4.0) in a fixed order (thread-strided partials, a fixed shuffle
//                            tree, the warps in order), and the order statistics at ranks floor((m - 1) * 0.95) and the
//                            next one by an 8-bit radix select over the 64-bit patterns (order-preserving for
//                            non-negative doubles), starting at the first byte where the smallest and the largest
//                            pattern differ.  Every step is deterministic: the outputs are bit-reproducible.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace octm {

constexpr int kSpThreads = 256;
constexpr int kSpTile = 16384;       // source vertices per sorted shared-memory tile (2 B each)
constexpr int kSpQueries = 8192;     // queries whose d2 stay in shared memory (8 B each); longer lists use d2

struct SpacingParams {
    const uint32_t* verts;   // [n][K][2][max_pts]
    const uint32_t* n_pts;   // [n][K][2]
    long long n_units;       // n * K * 2
    int max_pts;
    int ncol;                // doubled-lattice columns: x2 < ncol (2 W)
    int tile;                // source tile capacity
    int qcap;                // queries kept in shared memory (0: every unit stores to d2)
    double wy, wx;
    double* d2;              // [n][K][2][max_pts]
    double* max_sq;          // [n][K][2]
    double* p95_sq;          // [n][K][2][2]
    double* sum_dist;        // [n][K][2]
};

// One warp: the digit of rank `rank` among the 256 counts h[] and the rank left inside that digit.
__device__ __forceinline__ void radix_digit(const uint32_t* h, uint32_t rank, uint32_t& digit, uint32_t& rest) {
    const int lane = threadIdx.x & 31;
    uint32_t c[8], tot = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { c[j] = h[lane * 8 + j]; tot += c[j]; }
    uint32_t inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    const uint32_t exc = inc - tot;
    const bool mine = exc <= rank && rank < inc;               // exactly one lane
    const int owner = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
    uint32_t d = 0, r = rank - exc;
    if (mine) {
        for (int j = 0; j < 8; ++j) {
            if (r < c[j]) { d = lane * 8 + j; break; }
            r -= c[j];
        }
    }
    digit = __shfl_sync(0xffffffffu, d, owner);
    rest = __shfl_sync(0xffffffffu, r, owner);
}

__device__ __forceinline__ double scan_column(const uint16_t* ys, uint32_t lo, uint32_t hi, int qy, double wy, double wxb,
                                              double best) {
    for (uint32_t i = lo; i < hi; ++i) {
        const int a = static_cast<int>(ys[i]) - qy;
        best = fmin(best, __dadd_rn(__dmul_rn(wy, static_cast<double>(a * a)), wxb));
    }
    return best;
}

__global__ void __launch_bounds__(kSpThreads) distance_spacing_kernel(const SpacingParams p) {
    extern __shared__ __align__(16) uint8_t dsm[];
    __shared__ uint32_t s_hist[512];
    __shared__ uint32_t s_scan[33];
    __shared__ unsigned long long s_max[kSpThreads / 32], s_min[kSpThreads / 32];
    __shared__ double s_sum[kSpThreads / 32];
    __shared__ uint32_t s_sel[4];                  // digit and remaining rank of the low and the high order statistic
    double* const s_q = reinterpret_cast<double*>(dsm);                                          // qcap entries
    uint32_t* const col = reinterpret_cast<uint32_t*>(dsm + static_cast<size_t>(p.qcap) * 8);     // ncol + 1 entries
    uint16_t* const ys = reinterpret_cast<uint16_t*>(col + p.ncol + 1);                            // tile entries
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cap = p.max_pts, ncol = p.ncol;
    const int per = (ncol + kSpThreads - 1) / kSpThreads;       // columns per thread in the prefix sum

    for (long long unit = blockIdx.x; unit < p.n_units; unit += gridDim.x) {
        const long long pair = unit >> 1;
        const int dir = static_cast<int>(unit & 1);
        const int ns = static_cast<int>(min(p.n_pts[pair * 2 + dir], static_cast<uint32_t>(cap)));
        const int nq = static_cast<int>(min(p.n_pts[pair * 2 + 1 - dir], static_cast<uint32_t>(cap)));
        if (ns == 0 || nq == 0) {                  // CTA-uniform
            if (tid == 0) {
                p.max_sq[unit] = 0.0;
                p.p95_sq[unit * 2] = p.p95_sq[unit * 2 + 1] = 0.0;
                p.sum_dist[unit] = 0.0;
            }
            continue;
        }
        const uint32_t* vs = p.verts + (pair * 2 + dir) * static_cast<long long>(cap);
        const uint32_t* vq = p.verts + (pair * 2 + 1 - dir) * static_cast<long long>(cap);
        double* const dq = nq <= p.qcap ? s_q : p.d2 + unit * static_cast<long long>(cap);

        for (int t0 = 0; t0 < ns; t0 += p.tile) {
            const int nt = min(p.tile, ns - t0);
            __syncthreads();                       // the previous tile's (or unit's) readers are done
            for (int i = tid; i <= ncol; i += kSpThreads) col[i] = 0u;
            __syncthreads();
            // counting sort by column: count into col[x + 1] ...
            for (int i = tid; i < nt; i += kSpThreads) atomicAdd(&col[min(static_cast<int>(vs[t0 + i] & 0xffffu), ncol - 1) + 1], 1u);
            __syncthreads();
            {   // ... exclusive prefix sum in place (col[x + 1] = first slot of column x) ...
                const int b0 = 1 + tid * per;
                uint32_t s = 0, total;
                for (int k = 0; k < per; ++k)
                    if (b0 + k <= ncol) s += col[b0 + k];
                uint32_t off = block_excl_scan_sum<uint32_t>(s, s_scan, total);
                for (int k = 0; k < per; ++k)
                    if (b0 + k <= ncol) {
                        const uint32_t c = col[b0 + k];
                        col[b0 + k] = off;
                        off += c;
                    }
            }
            __syncthreads();
            // ... and scatter: afterwards col[x + 1] is the end of column x, so column x is col[x] .. col[x + 1]
            for (int i = tid; i < nt; i += kSpThreads) {
                const uint32_t v = vs[t0 + i];
                ys[atomicAdd(&col[min(static_cast<int>(v & 0xffffu), ncol - 1) + 1], 1u)] = static_cast<uint16_t>(v >> 16);
            }
            __syncthreads();
            for (int j = tid; j < nq; j += kSpThreads) {
                const uint32_t v = vq[j];
                const int qy = static_cast<int>(v >> 16), qx = static_cast<int>(v & 0xffffu);
                double best = t0 == 0 ? __longlong_as_double(0x7ff0000000000000ll) : dq[j];     // +inf
                for (int b = 0;; ++b) {
                    const double wxb = __dmul_rn(p.wx, static_cast<double>(b * b));
                    if (wxb > best) break;                 // no column this far or farther can hold a nearer vertex
                    const int cl = qx - b, cr = qx + b;
                    if (cl < 0 && cr >= ncol) break;
                    if (cl >= 0 && cl < ncol) best = scan_column(ys, col[cl], col[cl + 1], qy, p.wy, wxb, best);
                    if (b > 0 && cr < ncol) best = scan_column(ys, col[cr], col[cr + 1], qy, p.wy, wxb, best);
                }
                dq[j] = best;
            }
        }
        __syncthreads();                           // every query's d2 is written

        // max, min (of the bit patterns) and sum sqrt(d2 / 4.0): thread-strided, a fixed shuffle tree, warps in order
        unsigned long long vmax = 0ull, vmin = ~0ull;
        double ds = 0.0;
        for (int j = tid; j < nq; j += kSpThreads) {
            const double x = dq[j];
            const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(x));
            vmax = max(vmax, bits);
            vmin = min(vmin, bits);
            ds = __dadd_rn(ds, sqrt(x / 4.0));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
            vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
            ds = __dadd_rn(ds, __shfl_xor_sync(0xffffffffu, ds, o));
        }
        if (lane == 0) { s_max[warp] = vmax; s_min[warp] = vmin; s_sum[warp] = ds; }
        __syncthreads();
        vmax = s_max[0]; vmin = s_min[0]; ds = s_sum[0];
        for (int w = 1; w < kSpThreads / 32; ++w) {
            vmax = max(vmax, s_max[w]);
            vmin = min(vmin, s_min[w]);
            ds = __dadd_rn(ds, s_sum[w]);
        }

        // numpy linear percentile: virtual index (m - 1) * 0.95, neighbours floor and floor + 1
        const uint32_t r_lo = static_cast<uint32_t>(floor(__dmul_rn(static_cast<double>(nq - 1), 0.95)));
        uint32_t rl = r_lo, rh = r_lo + 1 < static_cast<uint32_t>(nq) ? r_lo + 1 : r_lo;
        unsigned long long pl = vmin, ph = vmin;
        if (vmin != vmax) {
            // every pattern lies between vmin and vmax, so all share the bits above the highest one where those differ
            int shift = (63 - __clzll(static_cast<long long>(vmin ^ vmax))) & ~7;
            pl = ph = shift == 56 ? 0ull : vmin >> (shift + 8);
            for (; shift >= 0; shift -= 8) {
                for (int i = tid; i < 512; i += kSpThreads) s_hist[i] = 0u;
                __syncthreads();
                // the loop bound is uniform over the CTA, so every warp is converged at the match
                for (int base = 0; base < nq; base += kSpThreads) {
                    const int j = base + tid;
                    uint32_t klo = 0xffffffffu, khi = 0xffffffffu;
                    if (j < nq) {
                        const unsigned long long x = static_cast<unsigned long long>(__double_as_longlong(dq[j]));
                        const unsigned long long top = shift == 56 ? 0ull : x >> (shift + 8);
                        const uint32_t d = static_cast<uint32_t>(x >> shift) & 0xffu;
                        if (top == pl) klo = d;
                        if (top == ph) khi = 256u + d;
                    }
                    const uint32_t mlo = __match_any_sync(0xffffffffu, klo), mhi = __match_any_sync(0xffffffffu, khi);
                    if (klo != 0xffffffffu && (mlo & lanemask_lt()) == 0) atomicAdd(&s_hist[klo], static_cast<uint32_t>(__popc(mlo)));
                    if (khi != 0xffffffffu && (mhi & lanemask_lt()) == 0) atomicAdd(&s_hist[khi], static_cast<uint32_t>(__popc(mhi)));
                }
                __syncthreads();
                if (warp == 0) {
                    uint32_t dl, ql, dh, qh;
                    radix_digit(s_hist, rl, dl, ql);
                    radix_digit(s_hist + 256, rh, dh, qh);
                    if (lane == 0) { s_sel[0] = dl; s_sel[1] = ql; s_sel[2] = dh; s_sel[3] = qh; }
                }
                __syncthreads();
                pl = (pl << 8) | s_sel[0];
                rl = s_sel[1];
                ph = (ph << 8) | s_sel[2];
                rh = s_sel[3];
            }
        }
        if (tid == 0) {
            p.max_sq[unit] = __longlong_as_double(static_cast<long long>(vmax));
            p.p95_sq[unit * 2 + 0] = __longlong_as_double(static_cast<long long>(pl));
            p.p95_sq[unit * 2 + 1] = __longlong_as_double(static_cast<long long>(ph));
            p.sum_dist[unit] = ds;
        }
    }
}

}  // namespace octm

// ----------------------------------------------------------------------------------- C ABI
extern "C" int octm_contour2d_distance_spacing(const uint32_t* verts, const uint32_t* n_pts, int64_t n_items,
                                               int num_classes, int max_pts, int H, int W, const double* spacing,
                                               double* max_sq, double* p95_sq, double* sum_dist, double* d2, int keep_d2,
                                               void* stream) {
    if (n_items < 0 || num_classes < 1 || max_pts < 8) return octm::fail(OCTM_ERR_INVALID, "bad shape");
    if (H < 1 || W < 1 || H > 8192 || W > 8192) return octm::fail(OCTM_ERR_INVALID, "H, W outside [1, 8192]");
    if (spacing == nullptr) return octm::fail(OCTM_ERR_INVALID, "null pointer: spacing");
    for (int a = 0; a < 2; ++a)
        if (!std::isfinite(spacing[a]) || !(spacing[a] > 0.0))
            return octm::fail(OCTM_ERR_INVALID, "spacing[%d] = %g: must be finite and > 0", a, spacing[a]);
    const double wy = spacing[0] * spacing[0], wx = spacing[1] * spacing[1];
    // the kernel works with the squares: each must be a normal double, and so must every q the image can hold
    for (int a = 0; a < 2; ++a)
        if (!std::isnormal(a == 0 ? wy : wx))
            return octm::fail(OCTM_ERR_INVALID, "spacing[%d] = %g: its square is not a normal double", a, spacing[a]);
    const double ry = 2.0 * H, rx = 2.0 * W;      // beyond every lattice offset of the image
    if (!std::isfinite(wy * (ry * ry) + wx * (rx * rx)))
        return octm::fail(OCTM_ERR_INVALID, "spacing: the squared diagonal of the image overflows a double");
    if (n_items == 0) return OCTM_OK;
    if (!verts || !n_pts || !max_sq || !p95_sq || !sum_dist) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    if (d2 == nullptr) return octm::fail(OCTM_ERR_INVALID, "d2 scratch [n][K][2][max_pts] (float64) is required");
    const int ncol = 2 * W;
    const int tile = std::min(max_pts, octm::kSpTile);
    const int qcap = keep_d2 ? 0 : std::min(max_pts, octm::kSpQueries);
    const size_t smem = static_cast<size_t>(qcap) * 8 + (static_cast<size_t>(ncol) + 1) * 4 + static_cast<size_t>(tile) * 2;
    if (smem + 8192 > static_cast<size_t>(octm::max_optin_smem()))
        return octm::fail(OCTM_ERR_UNSUPPORTED, "W = %d: the column table does not fit shared memory", W);
    if (cudaFuncSetAttribute(octm::distance_spacing_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem)) != cudaSuccess)
        return octm::fail(OCTM_ERR_LAUNCH, "cudaFuncSetAttribute(distance_spacing_kernel) failed");
    const long long n_units = n_items * num_classes * 2;
    octm::SpacingParams p{verts, n_pts, n_units, max_pts, ncol, tile, qcap, wy, wx, d2, max_sq, p95_sq, sum_dist};
    const long long grid = octm::resident_grid(n_units, octm::distance_spacing_kernel, octm::kSpThreads, smem, 1);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    OCTM_TIMED("distance_spacing_kernel", st)
        octm::distance_spacing_kernel<<<static_cast<unsigned>(grid), octm::kSpThreads, smem, st>>>(p);
    return octm::check_launch("distance_spacing_kernel");
}
