// Connected components of every class of a label map (build-defined, no reference counterpart) -- sm_100a.
//
// Per (item i, class c, map m; o the other map) and connectivity C in {4, 8}:
//     n_comp[i][c][m] = number of C-connected components of (L_m == c)      (scipy.ndimage.label)
//     n_hit[i][c][m]  = how many of them share at least one pixel with (L_o == c)
// Labels >= K belong to no class and are never counted.
//
//   components_kernel  one warp (= one CTA) per (item, map) walks the rows top to bottom with a union-find over RUNS,
//                      maximal horizontal stretches of equal labels.  Pixels join same-valued neighbours only, so the
//                      sets are the components of all K classes at once.  Per row:
//                      A  runs: a lane owns 16 columns of a 512-column pass; run starts (label changes) and hit pixels
//                         (L_m == L_o) become 16-bit masks, one warp scan of (popc starts | popc hits << 16) gives each
//                         run its index and the hit prefix at its start, so run r is hit iff hp[r + 1] > hp[r].
//                      B  link: run r joins every run of the previous row with its label whose columns meet
//                         [start, end) (widened by one column on each side for 8-connectivity): a binary search for
//                         the first candidate, then consecutive runs (runs partition a row).  The union is lock-free
//                         atomicMin on roots; this row's runs are nodes [0, W), the previous row's [W, 2W), so a set
//                         that continues into this row has a root in this row.
//                      C  hit flags of this row's runs and of merged previous sets are OR-ed into the new roots; a
//                         previous set whose root is still a previous-row node continues nowhere: it is closed and
//                         counted once into n_comp (and n_hit when flagged).
//                      D  this row becomes the previous row, re-rooted on its own run indices with flattened parents.
//                      After the last row every open set is counted.  State is O(W) per warp and sized for the worst
//                      case of one run per pixel, so any label map completes: no workspace, no bound, no retry.
#include "crack_masks.cuh"

namespace octm {

constexpr int kCcSeg = 512;              // columns per warp pass: 32 lanes x 16 labels
constexpr uint32_t kCcRoot = 1u << 31;   // prev_sl: the run is the root of its set

struct ComponentsParams {
    const uint8_t* yt;
    const uint8_t* yp;
    long long n_items;
    int H, W, K;
    int conn8;              // 1: 8-connectivity, 0: 4-connectivity
    uint32_t* n_comp;       // [n][K][2]
    uint32_t* n_hit;        // [n][K][2]
};

// shared memory of one warp, in words: parent [2W], cur_sl / prev_sl [W + 1] (start | label << 16, root bit in prev),
// cur_hp [W + 1] (hit prefix), flags of this / the previous row's runs [W / 32 + 1] each
__host__ __device__ inline size_t cc_smem_words(int W) {
    return 2 * static_cast<size_t>(W) + 3 * (static_cast<size_t>(W) + 1) + 2 * (static_cast<size_t>(W) / 32 + 1);
}

__device__ __forceinline__ uint32_t cc_find(const volatile uint32_t* par, uint32_t x) {
    uint32_t p = par[x];
    while (p != x) {
        x = p;
        p = par[x];
    }
    return x;
}

// union of the sets of a and b: the larger root is linked to the smaller (lock-free, any number of lanes at once)
__device__ __forceinline__ void cc_unite(uint32_t* par, uint32_t a, uint32_t b) {
    const volatile uint32_t* vp = par;
    while (true) {
        a = cc_find(vp, a);
        b = cc_find(vp, b);
        if (a == b) return;
        if (a > b) {
            const uint32_t t = a;
            a = b;
            b = t;
        }
        const uint32_t old = atomicMin(par + b, a);
        if (old == b) return;
        b = old;
    }
}

__device__ __forceinline__ uint32_t byte_of(const uint4& v, int i) {
    const uint32_t w = i < 4 ? v.x : i < 8 ? v.y : i < 12 ? v.z : v.w;
    return (w >> (8 * (i & 3))) & 0xffu;
}

template <bool VEC>
__global__ void __launch_bounds__(32) components_kernel(const ComponentsParams p) {
    extern __shared__ uint32_t sm[];
    __shared__ uint32_t s_cnt[OCTM_MAX_CLASSES][2];    // closed sets / closed hit sets per class
    const int lane = threadIdx.x;
    const int H = p.H, W = p.W, K = p.K;
    uint32_t* parent = sm;                             // [0, W): this row's runs, [W, 2W): the previous row's
    uint32_t* cur_sl = parent + 2 * W;
    uint32_t* prev_sl = cur_sl + W + 1;
    uint32_t* cur_hp = prev_sl + W + 1;
    uint32_t* cur_fl = cur_hp + W + 1;
    uint32_t* prev_fl = cur_fl + W / 32 + 1;
    const int nseg = (W + kCcSeg - 1) / kCcSeg;
    if (lane < OCTM_MAX_CLASSES) s_cnt[lane][0] = s_cnt[lane][1] = 0u;
    __syncwarp();

    const long long units = p.n_items * 2;
    for (long long unit = blockIdx.x; unit < units; unit += gridDim.x) {
        const long long item = unit >> 1;
        const int map = static_cast<int>(unit & 1);
        const long long off = item * static_cast<long long>(H) * W;
        const uint8_t* lm = (map ? p.yp : p.yt) + off;
        const uint8_t* lo = (map ? p.yt : p.yp) + off;
        auto count = [&](uint32_t label, bool hit) {
            if (label < static_cast<uint32_t>(K)) {
                atomicAdd(&s_cnt[label][0], 1u);
                if (hit) atomicAdd(&s_cnt[label][1], 1u);
            }
        };

        int nprev = 0;
        for (int y = 0; y < H; ++y) {
            const uint8_t* rm = lm + static_cast<long long>(y) * W;
            const uint8_t* ro = lo + static_cast<long long>(y) * W;
            // A: runs of this row
            uint32_t runs = 0, hits = 0, left = 0;
            for (int seg = 0; seg < nseg; ++seg) {
                const int col0 = seg * kCcSeg + lane * 16;
                const uint4 a = load16<VEC>(rm, col0, W);
                const uint4 b = load16<VEC>(ro, col0, W);
                uint32_t lb = __shfl_up_sync(kFull, a.w >> 24, 1);
                if (lane == 0) lb = left;
                const uint4 a0 = make_uint4((a.x << 8) | lb, __funnelshift_l(a.x, a.y, 8), __funnelshift_l(a.y, a.z, 8),
                                            __funnelshift_l(a.z, a.w, 8));     // labels of columns x - 1
                const int nv = min(max(W - col0, 0), 16);
                const uint32_t valid = (1u << nv) - 1u;
                uint32_t st = ~eq16(a, a0) & valid;
                if (col0 == 0) st |= 1u;
                const uint32_t hm = eq16(a, b) & valid;
                const uint32_t mine = __popc(st) | __popc(hm) << 16;
                uint32_t incl = mine;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t v = __shfl_up_sync(kFull, incl, o);
                    if (lane >= o) incl += v;
                }
                const uint32_t excl = incl - mine;
                uint32_t r = runs + (excl & 0xffffu);
                const uint32_t h0 = hits + (excl >> 16);
                for (uint32_t s = st; s != 0u; s &= s - 1u, ++r) {
                    const int i = __ffs(s) - 1;
                    cur_sl[r] = static_cast<uint32_t>(col0 + i) | byte_of(a, i) << 16;
                    cur_hp[r] = h0 + __popc(hm & ((1u << i) - 1u));
                }
                const uint32_t tot = __shfl_sync(kFull, incl, 31);
                runs += tot & 0xffffu;
                hits += tot >> 16;
                left = __shfl_sync(kFull, a.w >> 24, 31);
            }
            const int ncur = static_cast<int>(runs);
            if (lane == 0) {
                cur_sl[ncur] = static_cast<uint32_t>(W);
                cur_hp[ncur] = hits;
            }
            for (int r = lane; r < ncur; r += 32) parent[r] = static_cast<uint32_t>(r);
            for (int j = lane; j <= ncur / 32; j += 32) cur_fl[j] = 0u;
            __syncwarp();

            // B: link to the previous row
            for (int r = lane; r < ncur; r += 32) {
                const uint32_t sl = cur_sl[r], label = sl >> 16;
                if (label >= static_cast<uint32_t>(K) || nprev == 0) continue;
                const int ca = max(static_cast<int>(sl & 0xffffu) - p.conn8, 0);
                const int cb = min(static_cast<int>(cur_sl[r + 1] & 0xffffu) + p.conn8, W);      // [ca, cb)
                int lo_ = 0, hi_ = nprev - 1;                  // last previous run starting at or before ca
                while (lo_ < hi_) {
                    const int mid = (lo_ + hi_ + 1) >> 1;
                    if (static_cast<int>(prev_sl[mid] & 0xffffu) <= ca) lo_ = mid;
                    else hi_ = mid - 1;
                }
                for (int q = lo_; q < nprev; ++q) {
                    const uint32_t ps = prev_sl[q];
                    if (static_cast<int>(ps & 0xffffu) >= cb) break;
                    if (((ps >> 16) & 0xffu) == label) cc_unite(parent, static_cast<uint32_t>(r), static_cast<uint32_t>(W + q));
                }
            }
            __syncwarp();

            // C: hit flags into the new roots; close the previous sets that continue nowhere
            for (int r = lane; r < ncur; r += 32) {
                const uint32_t root = cc_find(parent, static_cast<uint32_t>(r));
                parent[r] = root;
                if (cur_hp[r + 1] > cur_hp[r]) atomicOr(cur_fl + (root >> 5), 1u << (root & 31));
            }
            for (int q = lane; q < nprev; q += 32) {
                const uint32_t ps = prev_sl[q];
                if (!(ps & kCcRoot)) continue;
                const bool flag = (prev_fl[q >> 5] >> (q & 31)) & 1u;
                const uint32_t root = cc_find(parent, static_cast<uint32_t>(W + q));
                if (root >= static_cast<uint32_t>(W)) count((ps >> 16) & 0xffu, flag);
                else if (flag) atomicOr(cur_fl + (root >> 5), 1u << (root & 31));
            }
            __syncwarp();

            // D: this row becomes the previous one
            for (int r = lane; r < ncur; r += 32) {
                const uint32_t root = parent[r];
                prev_sl[r] = cur_sl[r] | (root == static_cast<uint32_t>(r) ? kCcRoot : 0u);
                parent[W + r] = W + root;
            }
            for (int j = lane; j <= ncur / 32; j += 32) prev_fl[j] = cur_fl[j];
            if (lane == 0) prev_sl[ncur] = static_cast<uint32_t>(W);
            nprev = ncur;
            __syncwarp();
        }
        for (int q = lane; q < nprev; q += 32) {                // the sets still open after the last row
            const uint32_t ps = prev_sl[q];
            if (ps & kCcRoot) count((ps >> 16) & 0xffu, (prev_fl[q >> 5] >> (q & 31)) & 1u);
        }
        __syncwarp();
        if (lane < K) {
            const long long o = (item * K + lane) * 2 + map;
            p.n_comp[o] = s_cnt[lane][0];
            p.n_hit[o] = s_cnt[lane][1];
            s_cnt[lane][0] = s_cnt[lane][1] = 0u;
        }
        __syncwarp();
    }
}

}  // namespace octm

// ----------------------------------------------------------------------------------- C ABI
extern "C" int octm_components_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                  int num_classes, int connectivity, uint32_t* n_comp, uint32_t* n_hit, void* stream) {
    if (connectivity != 4 && connectivity != 8)
        return octm::fail(OCTM_ERR_INVALID, "connectivity %d is not 4 or 8", connectivity);
    if (int e = octm::check_shape(n_items, H, W, num_classes, 8)) return e;    // no vertex bound: 8 passes that check
    if (n_items == 0) return OCTM_OK;
    if (!y_true || !y_pred || !n_comp || !n_hit) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    const size_t smem = octm::cc_smem_words(W) * sizeof(uint32_t);
    if (smem + 1024 > static_cast<size_t>(octm::max_optin_smem()))
        return octm::fail(OCTM_ERR_UNSUPPORTED, "W = %d: the run state does not fit shared memory", W);
    octm::ComponentsParams p{};
    p.yt = y_true;
    p.yp = y_pred;
    p.n_items = n_items;
    p.H = H;
    p.W = W;
    p.K = num_classes;
    p.conn8 = connectivity == 8;
    p.n_comp = n_comp;
    p.n_hit = n_hit;
    const bool vec = W % 16 == 0 && reinterpret_cast<uintptr_t>(y_true) % 16 == 0 && reinterpret_cast<uintptr_t>(y_pred) % 16 == 0;
    auto kern = vec ? octm::components_kernel<true> : octm::components_kernel<false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
        return octm::fail(OCTM_ERR_LAUNCH, "cudaFuncSetAttribute(components_kernel) failed");
    const unsigned grid = static_cast<unsigned>(octm::resident_grid(n_items * 2, kern, 32, smem, 1));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OCTM_TIMED("components_kernel", s) kern<<<grid, 32, smem, s>>>(p);
    return octm::check_launch("components_kernel");
}
