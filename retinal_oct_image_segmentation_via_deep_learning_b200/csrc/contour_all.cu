// All-contour boundary vertices (build-defined extension of the contour metrics) -- sm_100a.
//
// The reference's contour metrics use contour [0] of find_contours(mask, 0.5) only (contour.cu).  This stage emits,
// for every class c of a label map, the vertex set of ALL its contours:
//     V(c) = doubled-lattice midpoints of every crack between two 4-adjacent pixels exactly one of which is class c
//          = unique(concatenate(find_contours(L == c, 0.5))) * 2
// each vertex once (no closing repeats).  A crack between labels a != b is one vertex of class a and one of class b.
// Lattice row 2y holds the cracks (y, x) | (y, x + 1) at x2 = 2x + 1, row 2y + 1 the cracks (y, x) | (y + 1, x) at
// x2 = 2x.  The vertices of a class are stored in raster order of the doubled lattice (row y2, then x2), so that the
// distance select kernel, which sums sqrt(D2 / 4) in query order, gives bit-reproducible sums.
//
//   contour_all_vertices_kernel  one CTA per (item, map), kAllWarps warps; an iteration reads kAllWarps image rows,
//                        warp w owns row y = y0 + w and with it lattice rows 2y and 2y + 1 (it reads rows y and y + 1).
//                        A lane holds 16 labels of each of the two rows; per class it forms a 16-bit mask of the
//                        horizontal and one of the vertical cracks it owns (byte compares in 32-bit words).  Pass 1
//                        counts (popc, warp sum), a shared-memory scan over the warps orders the rows, pass 2 writes
//                        at the running base of the class: first max_pts vertices stored, the count kept exact.
// The distance stage is the one of the contour [0] path (octm_contour2d_distance): it takes any vertex lists.
#include "crack_masks.cuh"

namespace octm {

constexpr int kAllWarps = 8;
constexpr int kAllSeg = 512;          // columns per warp pass: 32 lanes x 16 labels

struct AllVertsParams {
    const uint8_t* yt;
    const uint8_t* yp;
    long long n_items;
    int H, W, K, max_pts;
    uint32_t* verts;     // [n][K][2][max_pts]
    uint32_t* n_pts;     // [n][K][2]
    uint32_t* flags;     // [n][K], zeroed by the caller
};

template <bool VEC>
__global__ void __launch_bounds__(kAllWarps * 32, 3) contour_all_vertices_kernel(const AllVertsParams p) {
    __shared__ uint32_t s_cnt[2][kAllWarps][OCTM_MAX_CLASSES];     // per warp and class: even | odd << 16 (double-buffered)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int H = p.H, W = p.W, K = p.K;
    const int nseg = (W + kAllSeg - 1) / kAllSeg;
    const uint32_t cap = static_cast<uint32_t>(p.max_pts);
    for (long long unit = blockIdx.x; unit < p.n_items * 2; unit += gridDim.x) {
        const long long item = unit >> 1;
        const int map = static_cast<int>(unit & 1);
        const uint8_t* img = (map ? p.yp : p.yt) + item * static_cast<long long>(H) * W;
        uint32_t run = 0;          // lanes c and 16 + c: vertices of class c in the rows of earlier iterations
        int buf = 0;
        for (int y0 = 0; y0 < H; y0 += kAllWarps, buf ^= 1) {
            const int y = y0 + warp;
            const uint8_t* ra = img + static_cast<long long>(y) * W;
            const uint8_t* rb = y + 1 < H ? ra + W : nullptr;
            uint32_t m[OCTM_MAX_CLASSES];
            bool cached = false;   // single segment: the masks of pass 1 are reused by pass 2
            uint32_t cnt = 0;      // lane c: this warp's even | odd << 16 count of class c
            if (y < H) {
                for (int seg = 0; seg < nseg; ++seg) {
                    if (!crack_masks<VEC>(ra, rb, seg * kAllSeg + lane * 16, W, K, lane, m)) continue;
                    cached = true;
#pragma unroll
                    for (int c = 0; c < OCTM_MAX_CLASSES; ++c) {
                        if (c >= K) break;
                        // at most 8191 / 8192 cracks per lattice row and class: the halves cannot carry
                        const uint32_t tot = __reduce_add_sync(kFull, __popc(m[c] & 0xffffu) | __popc(m[c] >> 16) << 16);
                        if (lane == c) cnt += tot;
                    }
                }
            }
            if (lane < OCTM_MAX_CLASSES) s_cnt[buf][warp][lane] = cnt;
            __syncthreads();
            // lanes c / 16 + c: where this warp's even / odd lattice row of class c starts
            const int c_own = lane & (OCTM_MAX_CLASSES - 1);
            uint32_t before = 0, total = 0;
#pragma unroll
            for (int w2 = 0; w2 < kAllWarps; ++w2) {
                const uint32_t v = s_cnt[buf][w2][c_own];
                const uint32_t s = (v & 0xffffu) + (v >> 16);
                before += w2 < warp ? s : 0u;
                total += s;
            }
            uint32_t base = run + before + (lane >= OCTM_MAX_CLASSES ? (s_cnt[buf][warp][c_own] & 0xffffu) : 0u);
            run += total;
            if (y >= H || !cached) continue;
            for (int seg = 0; seg < nseg; ++seg) {
                const int col0 = seg * kAllSeg + lane * 16;
                if (nseg > 1 && !crack_masks<VEC>(ra, rb, col0, W, K, lane, m)) continue;
#pragma unroll
                for (int c = 0; c < OCTM_MAX_CLASSES; ++c) {
                    if (c >= K) break;
                    const uint32_t own = __popc(m[c] & 0xffffu) | __popc(m[c] >> 16) << 16;
                    uint32_t incl = own;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t t = __shfl_up_sync(kFull, incl, o);
                        if (lane >= o) incl += t;
                    }
                    const uint32_t tot = __shfl_sync(kFull, incl, 31);
                    const uint32_t excl = incl - own;
                    uint32_t* out = p.verts + ((item * K + c) * 2 + map) * static_cast<long long>(cap);
                    uint32_t idx = __shfl_sync(kFull, base, c) + (excl & 0xffffu);
                    const uint32_t row_e = static_cast<uint32_t>(2 * y) << 16;
                    for (uint32_t bits = m[c] & 0xffffu; bits != 0u; bits &= bits - 1u, ++idx)
                        if (idx < cap) out[idx] = row_e | static_cast<uint32_t>(2 * (col0 + __ffs(bits) - 1) + 1);
                    idx = __shfl_sync(kFull, base, OCTM_MAX_CLASSES + c) + (excl >> 16);
                    const uint32_t row_o = static_cast<uint32_t>(2 * y + 1) << 16;
                    for (uint32_t bits = m[c] >> 16; bits != 0u; bits &= bits - 1u, ++idx)
                        if (idx < cap) out[idx] = row_o | static_cast<uint32_t>(2 * (col0 + __ffs(bits) - 1));
                    if (lane == c) base += tot & 0xffffu;
                    if (lane == OCTM_MAX_CLASSES + c) base += tot >> 16;
                }
            }
        }
        if (warp == 0 && lane < K) {
            p.n_pts[(item * K + lane) * 2 + map] = run;
            if (run > cap) atomicOr(p.flags + item * K + lane, map ? OCTM_CF_PRED_OVERFLOW : OCTM_CF_TRUE_OVERFLOW);
        }
        __syncthreads();           // s_cnt is reused by the next unit
    }
}

}  // namespace octm

// ----------------------------------------------------------------------------------- C ABI
extern "C" int octm_contour2d_all_vertices_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                              int num_classes, int max_pts, uint32_t* verts, uint32_t* n_pts,
                                              uint32_t* flags, void* stream) {
    if (int e = octm::check_shape(n_items, H, W, num_classes, max_pts)) return e;
    if (n_items == 0) return OCTM_OK;
    if (!y_true || !y_pred || !verts || !n_pts || !flags) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (cudaMemsetAsync(flags, 0, sizeof(uint32_t) * n_items * num_classes, s) != cudaSuccess)
        return octm::fail(OCTM_ERR_LAUNCH, "memset(flags) failed");
    const octm::AllVertsParams p{y_true, y_pred, n_items, H, W, num_classes, max_pts, verts, n_pts, flags};
    const bool vec = W % 16 == 0 && reinterpret_cast<uintptr_t>(y_true) % 16 == 0 && reinterpret_cast<uintptr_t>(y_pred) % 16 == 0;
    const long long units = n_items * 2;
    const unsigned grid = static_cast<unsigned>(units < (1ll << 30) ? units : (1ll << 30));
    if (vec) OCTM_TIMED("contour_all_vertices_kernel", s) octm::contour_all_vertices_kernel<true><<<grid, octm::kAllWarps * 32, 0, s>>>(p);
    else OCTM_TIMED("contour_all_vertices_kernel", s) octm::contour_all_vertices_kernel<false><<<grid, octm::kAllWarps * 32, 0, s>>>(p);
    return octm::check_launch("contour_all_vertices_kernel");
}

extern "C" int octm_contour2d_all_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                     int num_classes, int max_pts, uint32_t* n_pts, uint32_t* flags, uint32_t* max_sq,
                                     uint32_t* p95_sq, double* sum_dist, void* workspace, size_t workspace_bytes,
                                     void* stream) {
    if (int e = octm::check_shape(n_items, H, W, num_classes, max_pts)) return e;
    if (n_items == 0) return OCTM_OK;
    if (!y_true || !y_pred || !n_pts || !flags || !max_sq || !p95_sq || !sum_dist)
        return octm::fail(OCTM_ERR_INVALID, "null pointer");
    const size_t need = octm_contour2d_workspace_bytes(n_items, H, W, num_classes, max_pts);
    if (workspace == nullptr || workspace_bytes < need) return octm::fail(OCTM_ERR_WORKSPACE, "workspace too small: need %zu B", need);
    const octm::ContourWorkspace ws = octm::contour_workspace(n_items, num_classes, max_pts, workspace);
    if (int e = octm_contour2d_all_vertices_u8(y_true, y_pred, n_items, H, W, num_classes, max_pts, ws.verts, n_pts, flags, stream))
        return e;
    return octm_contour2d_distance(ws.verts, n_pts, n_items, num_classes, max_pts, H, W, max_sq, p95_sq, sum_dist, ws.d2, 0, stream);
}
