// Normalized surface Dice at tolerance tau (build-defined, no reference counterpart) -- sm_100a.
//
// Per (item i, class c) the surfaces are the all-contour vertex sets of contour_all.cu: V_t of (y_true == c) and V_p of
// (y_pred == c), every crack between two 4-adjacent pixels exactly one of which is class c, on the doubled lattice
// (row 2y: horizontal cracks at x2 = 2x + 1, row 2y + 1: vertical cracks at x2 = 2x).  For each integer threshold T_j
// (T_j = the largest D with sqrt(D / 4) <= tau_j, computed by the caller) the kernel counts
//     n_within[i][c][0][j] = #{ v in V_p : min_{u in V_t} |v - u|^2 <= T_j }      (direction 0: pred -> true)
//     n_within[i][c][1][j] = #{ v in V_t : min_{u in V_p} |v - u|^2 <= T_j }      (direction 1: true -> pred)
// and n_surf[i][c] = (|V_t|, |V_p|).  No vertex list and no nearest-neighbour search: only "is there a source vertex
// within T_j".
//
// Exactness.  A source vertex at offset (dy, dx) from a query vertex has dy^2 + dx^2 <= T_j only if |dy| <= R =
// floor(sqrt(T_max)) and, for that dy, |dx| <= r(dy) = floor(sqrt(T_j - dy^2)).  The kernel scans exactly these
// windows, every lattice row dy in [-R, R] and in it every column within r(dy), so each count is exact: no cap, no
// approximation.  Every vertex pair has dy == dx (mod 2) (y2 + x2 is odd for every vertex), so a row of the query's own
// parity is met at even dx = 2d, |d| <= r / 2, and a row of the other parity at odd dx: a horizontal-crack query
// (x2 = 2x + 1) meets a vertical-crack row (x2' = 2x') at dx = 2d - 1, d in [-(r - 1) / 2, (r + 1) / 2], and a
// vertical-crack query meets a horizontal-crack row at dx = 2d + 1, d in [-(r + 1) / 2, (r - 1) / 2] (d = x' - x in
// image columns).  T <= 256 (tau <= 8 px) gives R <= 16 lattice rows and |d| <= 8 columns.
//
//   surface_dice_kernel  one CTA of kSdWarps warps per (item, class group); an iteration handles kSdWarps image rows.
//                        A lane owns 16 columns and, per class and map, one crack word (crack_masks.cuh: 16 horizontal |
//                        16 vertical crack bits).  Shared memory holds a ring of these words for both maps: the
//                        iteration's rows plus a halo of ceil(R / 2) image rows on each side, so each label map is read
//                        once.  Warp w queries image row y0 + w: for every lattice row offset it dilates the other map's
//                        row words (a 48-bit window over the lane's word and its two neighbours) by the reach of each
//                        threshold with two shifted ORs of a power-of-two run mask, ORs the hits of the query bits,
//                        and finally popc + warp sum + one shared atomic per (class, direction, threshold).  A warp
//                        whose query words of a class are all zero skips the class (the common case on layers).
#include "crack_masks.cuh"

namespace octm {

constexpr int kSdWarps = 8;
constexpr int kSdSeg = 512;           // columns per warp pass: 32 lanes x 16 labels
constexpr int kSdMaxReach = 16;       // floor(sqrt(OCTM_SURFACE_DICE_MAX_SQ))

struct SurfaceDiceParams {
    const uint8_t* yt;
    const uint8_t* yp;
    long long n_items;
    int H, W, K;
    int group, n_groups;  // classes per CTA, class groups per item
    int n_thr;
    uint32_t thr[OCTM_SURFACE_DICE_MAX_TOL];   // ascending
    int reach;            // R = floor(sqrt(thr[n_thr - 1])) lattice rows
    int halo;             // ceil(R / 2) image rows
    int slots;            // ring rows: kSdWarps + 2 * halo
    int nw;               // crack words per row: 32 per 512-column segment
    uint32_t* n_surf;     // [n][K][2]
    uint32_t* n_within;   // [n][K][2][n_thr]
};

__device__ __forceinline__ int isqrt_small(int v) {      // floor(sqrt(v)), 0 <= v <= 256
    int r = static_cast<int>(sqrtf(static_cast<float>(v)));
    while (r * r > v) --r;
    while ((r + 1) * (r + 1) <= v) ++r;
    return r;
}

// Shift code of (query row type qt, |dy|, threshold j): the dilation by columns [lo, hi] of a source row is
// (x_p >> (16 + lo)) | (x_p >> (16 + hi - p + 1)), x_p the run-of-p mask of the 48-bit window, p = 2^psel the largest
// power of two <= hi - lo + 1.  Code = sh1 | sh2 << 8 | psel << 16 | 1 << 24; 0 = no source column within reach.
__device__ uint32_t range_code(int qt, int a, uint32_t T) {
    const int a2 = a * a;
    if (static_cast<uint32_t>(a2) > T) return 0u;
    const int r = isqrt_small(static_cast<int>(T) - a2);
    int lo, hi;
    if ((a & 1) == 0) {                 // same row type: dx = 2d
        lo = -(r >> 1);
        hi = r >> 1;
    } else {                            // other row type: dx odd
        if (r < 1) return 0u;
        lo = qt == 0 ? -((r - 1) >> 1) : -((r + 1) >> 1);
        hi = qt == 0 ? (r + 1) >> 1 : (r - 1) >> 1;
    }
    const int len = hi - lo + 1;
    const int psel = 31 - __clz(len);
    return static_cast<uint32_t>(16 + lo) | static_cast<uint32_t>(16 + hi - (1 << psel) + 1) << 8 |
           static_cast<uint32_t>(psel) << 16 | 1u << 24;
}

template <bool VEC>
__global__ void __launch_bounds__(kSdWarps * 32) surface_dice_kernel(const SurfaceDiceParams p) {
    extern __shared__ uint32_t ring[];   // [slots][2 maps][group][nw + 2]: one zero pad word at each end of a row
    __shared__ uint32_t s_code[2][kSdMaxReach + 1][OCTM_SURFACE_DICE_MAX_TOL];
    __shared__ uint32_t s_within[OCTM_MAX_CLASSES][2][OCTM_SURFACE_DICE_MAX_TOL];
    __shared__ uint32_t s_surf[OCTM_MAX_CLASSES][2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int H = p.H, W = p.W, K = p.K, G = p.group, n_thr = p.n_thr, R = p.reach;
    const int stride = p.nw + 2;
    const int nseg = (W + kSdSeg - 1) / kSdSeg;
    for (int e = tid; e < 2 * (kSdMaxReach + 1) * OCTM_SURFACE_DICE_MAX_TOL; e += blockDim.x) {
        const int j = e % OCTM_SURFACE_DICE_MAX_TOL, a = (e / OCTM_SURFACE_DICE_MAX_TOL) % (kSdMaxReach + 1);
        const int qt = e / (OCTM_SURFACE_DICE_MAX_TOL * (kSdMaxReach + 1));
        const uint32_t T = j == 0 ? p.thr[0] : j == 1 ? p.thr[1] : j == 2 ? p.thr[2] : p.thr[3];   // no local copy of p
        s_code[qt][a][j] = j < n_thr ? range_code(qt, a, T) : 0u;
    }
    for (int e = tid; e < p.slots * 2 * G * stride; e += blockDim.x) ring[e] = 0u;    // the pad words stay zero
    for (int e = tid; e < OCTM_MAX_CLASSES * 2 * OCTM_SURFACE_DICE_MAX_TOL; e += blockDim.x) (&s_within[0][0][0])[e] = 0u;
    if (tid < OCTM_MAX_CLASSES * 2) (&s_surf[0][0])[tid] = 0u;
    __syncthreads();

    const long long units = p.n_items * p.n_groups;
    for (long long unit = blockIdx.x; unit < units; unit += gridDim.x) {
        const long long item = unit / p.n_groups;
        const int g0 = static_cast<int>(unit % p.n_groups) * G;
        const int gk = min(G, K - g0);
        const long long off = item * static_cast<long long>(H) * W;

        // crack words of image row y (< H) of both maps, classes [g0, g0 + gk), into ring row y % slots
        auto load_row = [&](int y) {
            uint32_t* dst = ring + static_cast<size_t>(y % p.slots) * 2 * G * stride + 1;
#pragma unroll 1
            for (int map = 0; map < 2; ++map) {
                const uint8_t* ra = (map ? p.yp : p.yt) + off + static_cast<long long>(y) * W;
                const uint8_t* rb = y + 1 < H ? ra + W : nullptr;
                uint32_t* dm = dst + map * G * stride;
                for (int seg = 0; seg < nseg; ++seg) {
                    const int wi = seg * 32 + lane;
                    uint32_t m[OCTM_MAX_CLASSES];
                    const bool any = crack_masks<VEC>(ra, rb, seg * kSdSeg + lane * 16, W, g0 + gk, lane, m);
#pragma unroll
                    for (int c = 0; c < OCTM_MAX_CLASSES; ++c)
                        if (c >= g0 && c < g0 + gk) dm[(c - g0) * stride + wi] = any ? m[c] : 0u;
                }
            }
        };

        if (warp < p.halo && warp < H) load_row(warp);
        for (int y0 = 0; y0 < H; y0 += kSdWarps) {
            if (y0 + p.halo + warp < H) load_row(y0 + p.halo + warp);
            __syncthreads();
            const int y = y0 + warp;
            if (y < H) {
                const int ys = y % p.slots;
                const uint32_t* qrow = ring + static_cast<size_t>(ys) * 2 * G * stride + 1;
                for (int seg = 0; seg < nseg; ++seg) {
                    const int wi = seg * 32 + lane;
                    for (int g = 0; g < gk; ++g) {
#pragma unroll 1
                        for (int d = 0; d < 2; ++d) {          // direction 0: pred vertices -> true set; 1: true -> pred
                            const int qm = 1 - d, sm = d;
                            const uint32_t qword = qrow[(qm * G + g) * stride + wi];
                            if (!__any_sync(kFull, qword != 0u)) continue;
                            const uint32_t ns = __reduce_add_sync(kFull, __popc(qword));
                            if (lane == 0) atomicAdd(&s_surf[g][qm], ns);
                            uint32_t hit[OCTM_SURFACE_DICE_MAX_TOL] = {0u, 0u, 0u, 0u};
#pragma unroll
                            for (int qt = 0; qt < 2; ++qt) {
                                const uint32_t qbits = (qword >> (16 * qt)) & 0xffffu;
                                if (!__any_sync(kFull, qbits != 0u)) continue;
                                for (int dy = -R; dy <= R; ++dy) {
                                    const int sy2 = 2 * y + qt + dy;
                                    if (sy2 < 0 || (sy2 >> 1) >= H || qbits == 0u) continue;
                                    const int sh = 16 * (sy2 & 1);
                                    int slot = ys + (sy2 >> 1) - y;                 // (sy2 >> 1) % slots
                                    slot += slot < 0 ? p.slots : slot >= p.slots ? -p.slots : 0;
                                    const uint32_t* src = ring + static_cast<size_t>(slot) * 2 * G * stride + (sm * G + g) * stride + 1 + wi;
                                    const uint64_t win = static_cast<uint64_t>((src[-1] >> sh) & 0xffffu) |
                                                         static_cast<uint64_t>((src[0] >> sh) & 0xffffu) << 16 |
                                                         static_cast<uint64_t>((src[1] >> sh) & 0xffffu) << 32;
                                    if (win == 0u) continue;
                                    // run_p bit i = OR of window bits [i, i + p)
                                    const uint64_t run2 = win | win >> 1, run4 = run2 | run2 >> 2, run8 = run4 | run4 >> 4;
                                    const uint64_t run16 = run8 | run8 >> 8;
                                    const int a = dy < 0 ? -dy : dy;
#pragma unroll
                                    for (int j = 0; j < OCTM_SURFACE_DICE_MAX_TOL; ++j) {
                                        const uint32_t code = s_code[qt][a][j];
                                        if (code == 0u) continue;
                                        const uint32_t ps = (code >> 16) & 0xffu;
                                        const uint64_t xp = ps == 0 ? win : ps == 1 ? run2 : ps == 2 ? run4 : ps == 3 ? run8 : run16;
                                        const uint32_t dil = static_cast<uint32_t>(xp >> (code & 0xffu)) |
                                                             static_cast<uint32_t>(xp >> ((code >> 8) & 0xffu));
                                        hit[j] |= (qbits & dil) << (16 * qt);
                                    }
                                }
                            }
#pragma unroll
                            for (int j = 0; j < OCTM_SURFACE_DICE_MAX_TOL; ++j) {
                                if (j >= n_thr) break;
                                const uint32_t nh = __reduce_add_sync(kFull, __popc(hit[j]));
                                if (lane == 0 && nh != 0u) atomicAdd(&s_within[g][d][j], nh);
                            }
                        }
                    }
                }
            }
            __syncthreads();           // the next iteration's loads overwrite ring rows this one read
        }
        if (tid < gk * 2) {
            const int g = tid >> 1, m = tid & 1;
            p.n_surf[(item * K + g0 + g) * 2 + m] = s_surf[g][m];
            s_surf[g][m] = 0u;
        }
        if (tid < gk * 2 * n_thr) {
            const int j = tid % n_thr, d = (tid / n_thr) & 1, g = tid / (2 * n_thr);
            p.n_within[((item * K + g0 + g) * 2 + d) * n_thr + j] = s_within[g][d][j];
            s_within[g][d][j] = 0u;
        }
        // the zeroing above precedes the next unit's atomics: those follow its first __syncthreads
    }
}

}  // namespace octm

// ----------------------------------------------------------------------------------- C ABI
extern "C" int octm_surface_dice_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                    int num_classes, const uint32_t* thresholds_sq, int n_thresholds, uint32_t* n_surf,
                                    uint32_t* n_within, void* stream) {
    if (int e = octm::check_shape(n_items, H, W, num_classes, 8)) return e;    // no vertex bound: 8 passes that check
    if (thresholds_sq == nullptr) return octm::fail(OCTM_ERR_INVALID, "null pointer: thresholds_sq");
    if (n_thresholds < 1 || n_thresholds > OCTM_SURFACE_DICE_MAX_TOL)
        return octm::fail(OCTM_ERR_INVALID, "n_thresholds %d outside [1, %d]", n_thresholds, OCTM_SURFACE_DICE_MAX_TOL);
    octm::SurfaceDiceParams p{};
    for (int j = 0; j < n_thresholds; ++j) {
        const uint32_t t = thresholds_sq[j];
        if (t > OCTM_SURFACE_DICE_MAX_SQ)
            return octm::fail(OCTM_ERR_INVALID, "thresholds_sq[%d] = %u > %d", j, t, OCTM_SURFACE_DICE_MAX_SQ);
        if (j > 0 && t < thresholds_sq[j - 1]) return octm::fail(OCTM_ERR_INVALID, "thresholds_sq not ascending");
        p.thr[j] = t;
    }
    if (n_items == 0) return OCTM_OK;
    if (!y_true || !y_pred || !n_surf || !n_within) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    int reach = 0;
    while ((reach + 1) * (reach + 1) <= static_cast<int>(p.thr[n_thresholds - 1])) ++reach;
    const int halo = (reach + 1) / 2, slots = octm::kSdWarps + 2 * halo;
    const int nw = (W + octm::kSdSeg - 1) / octm::kSdSeg * 32;
    const size_t per_class = static_cast<size_t>(slots) * 2 * (nw + 2) * sizeof(uint32_t);
    const size_t budget = static_cast<size_t>(octm::max_optin_smem()) - 4096;     // static shared memory + slack
    int group = static_cast<int>(budget / per_class < static_cast<size_t>(num_classes) ? budget / per_class : num_classes);
    if (group < 1) return octm::fail(OCTM_ERR_UNSUPPORTED, "W = %d: one class's ring does not fit shared memory", W);
    const int n_groups = (num_classes + group - 1) / group;
    group = (num_classes + n_groups - 1) / n_groups;
    const size_t smem = per_class * group;
    p.yt = y_true;
    p.yp = y_pred;
    p.n_items = n_items;
    p.H = H;
    p.W = W;
    p.K = num_classes;
    p.group = group;
    p.n_groups = n_groups;
    p.n_thr = n_thresholds;
    p.reach = reach;
    p.halo = halo;
    p.slots = slots;
    p.nw = nw;
    p.n_surf = n_surf;
    p.n_within = n_within;
    const bool vec = W % 16 == 0 && reinterpret_cast<uintptr_t>(y_true) % 16 == 0 && reinterpret_cast<uintptr_t>(y_pred) % 16 == 0;
    auto kern = vec ? octm::surface_dice_kernel<true> : octm::surface_dice_kernel<false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
        return octm::fail(OCTM_ERR_LAUNCH, "cudaFuncSetAttribute(surface_dice_kernel) failed");
    const long long units = n_items * n_groups;
    const unsigned grid = static_cast<unsigned>(octm::resident_grid(units, kern, octm::kSdWarps * 32, smem, 1));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OCTM_TIMED("surface_dice_kernel", s) kern<<<grid, octm::kSdWarps * 32, smem, s>>>(p);
    return octm::check_launch("surface_dice_kernel");
}
