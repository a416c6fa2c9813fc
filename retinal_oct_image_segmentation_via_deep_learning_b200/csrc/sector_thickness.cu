// Per-sector layer thickness of OCT volumes from the label pass's boundary rows -- sm_100a.
//
// The boundary rows are counts, b_k(x) = #{y : L[y][x] < k} (k = 1 .. K-1; b_0 = 0, b_K = H), so the thickness of the
// classes first .. last in A-scan x is b_{last+1}(x) - b_first(x) for any label map, layered or not.  A volume is
// items_per_volume consecutive items; every A-scan (item, x) carries a region code.  Per (volume, group, region) the
// kernel sums, over the A-scans of that region, the five integers
//     n, t, p, |t - p|, (t - p)^2            (t, p: group thickness of y_true / y_pred in pixels)
// exactly in int64 (the host checks items_per_volume * W * H^2 < 2^53), so the order of the atomics does not matter and
// the outputs are bit-reproducible.
//
//   sector_thickness_kernel  grid (chunks, volumes); one thread per A-scan of a chunk, groups in an inner loop.  The
//                            lanes of a warp with equal region codes (long runs in practice) are found with
//                            __match_any_sync and their values summed with __reduce_add_sync over that mask; the
//                            lowest lane adds the sums to the CTA's counters in shared memory, which are flushed to
//                            global memory once per CTA.  The shared counters are 32-bit words with a high word each:
//                            a 64-bit shared atomic is a compare-and-swap loop, which every warp of a CTA would retry
//                            on the same few counters, while a 32-bit add is native and its return value tells the one
//                            add that wraps the low word to carry into the high word, so the count stays exact.  Per lane t, p, |t - p| <= H and 32 H < 2^32; (t - p)^2 < 2^32
//                            summed over 32 lanes stays below 2^32 only while H <= 8192, so taller maps reduce it in
//                            three 21-bit limbs (kWide).
#include <algorithm>

#include "common.cuh"

namespace octm {

constexpr int kStThreads = 256;
constexpr int kStMaxGroups = 16;
constexpr int kStMaxRegions = 16;
constexpr int kStStats = 5;
// A-scans per CTA at most: two iterations of the CTA.  Chunks of 2,048 left 1.2-1.4 waves of CTAs on a B200 for
// 64-volume batches; chunks of 512 give 5 or more and took 17-22 % less time (DESIGN.md).
constexpr int kStMaxChunk = kStThreads * 2;

struct SectorParams {
    const int32_t* bnd_true;    // [n][K-1][W]
    const int32_t* bnd_pred;
    const uint8_t* region;      // [n][W]
    unsigned long long* sums;   // [V][G][R][5]
    int32_t* thick;             // [n][2][G][W] or null
    long long ascans;           // A-scans per volume: items_per_volume * W
    int items_per_volume;
    int K, H, W;
    int n_regions, n_groups;
    int chunk;                  // A-scans per CTA, a multiple of kStThreads
    unsigned long long first, last;     // group g's first / last class in bits 4g .. 4g + 3 (no local-memory copy)
};

// b_k of row pointer `rows` ([K-1][W] at column x): 0 for k = 0, H for k = K
__device__ __forceinline__ int boundary_at(const int32_t* rows, int k, int K, int H, int W) {
    return k == 0 ? 0 : k == K ? H : __ldg(rows + static_cast<long long>(k - 1) * W);
}

// Exact 64-bit add to a (lo, hi) pair of 32-bit shared counters: the add that wraps lo carries into hi.
__device__ __forceinline__ void add_wide(uint32_t* lo, uint32_t* hi, unsigned long long v) {
    const uint32_t vl = static_cast<uint32_t>(v);
    const uint32_t old = atomicAdd(lo, vl);
    const uint32_t up = static_cast<uint32_t>(v >> 32) + (old + vl < old ? 1u : 0u);
    if (up != 0u) atomicAdd(hi, up);
}

template <bool kWide>
__global__ void __launch_bounds__(kStThreads) sector_thickness_kernel(const SectorParams p) {
    constexpr int kSums = kStStats - 1;                     // sum t, sum p, sum |t - p|, sum (t - p)^2
    __shared__ uint32_t s_lo[kStMaxGroups * kStMaxRegions * kSums], s_hi[kStMaxGroups * kStMaxRegions * kSums];
    __shared__ uint32_t s_cnt[kStMaxRegions];               // A-scans per region: the same for every group
    const int nsum = p.n_groups * p.n_regions * kSums;
    for (int i = threadIdx.x; i < nsum; i += kStThreads) s_lo[i] = s_hi[i] = 0u;
    if (threadIdx.x < kStMaxRegions) s_cnt[threadIdx.x] = 0u;
    __syncthreads();

    const long long vol = blockIdx.y;
    const long long a0 = static_cast<long long>(blockIdx.x) * p.chunk;
    const long long a1 = min(a0 + p.chunk, p.ascans);
    // the loop bound is uniform over the CTA, so every warp is converged at the match and the reductions
    for (long long base = a0; base < a1; base += kStThreads) {
        const long long a = base + threadIdx.x;
        const bool valid = a < a1;
        long long item = 0;
        int x = 0;
        uint32_t key = 0xffffffffu;
        if (valid) {
            if (p.ascans <= 0xffffffffll) {                 // uniform: 32-bit division when the volume allows it
                const uint32_t a32 = static_cast<uint32_t>(a), w32 = static_cast<uint32_t>(p.W);
                const uint32_t il = a32 / w32;
                item = vol * p.items_per_volume + il;
                x = static_cast<int>(a32 - il * w32);
            } else {
                item = vol * p.items_per_volume + a / p.W;
                x = static_cast<int>(a % p.W);
            }
            const uint32_t r = p.region[item * p.W + x];
            if (r < static_cast<uint32_t>(p.n_regions)) key = r;
        }
        const uint32_t mask = __match_any_sync(0xffffffffu, key);
        const bool leader = key != 0xffffffffu && (mask & lanemask_lt()) == 0;
        if (leader) atomicAdd(&s_cnt[key], static_cast<uint32_t>(__popc(mask)));
        const long long row0 = item * (p.K - 1) * static_cast<long long>(p.W) + x;
        const int32_t* bt = p.bnd_true + row0;
        const int32_t* bp = p.bnd_pred + row0;
        int prev_l = -1, prev_t = 0, prev_q = 0;          // b_l of the previous group: groups often tile the classes
        for (int g = 0; g < p.n_groups; ++g) {
            int t = 0, q = 0;
            if (valid) {
                const int f = static_cast<int>((p.first >> (4 * g)) & 15ull);
                const int l = static_cast<int>((p.last >> (4 * g)) & 15ull) + 1;
                const int tf = f == prev_l ? prev_t : boundary_at(bt, f, p.K, p.H, p.W);
                const int qf = f == prev_l ? prev_q : boundary_at(bp, f, p.K, p.H, p.W);
                prev_l = l;
                prev_t = boundary_at(bt, l, p.K, p.H, p.W);
                prev_q = boundary_at(bp, l, p.K, p.H, p.W);
                t = prev_t - tf;
                q = prev_q - qf;
                if (p.thick != nullptr) {
                    int32_t* out = p.thick + (item * 2 * p.n_groups + g) * static_cast<long long>(p.W) + x;
                    out[0] = t;
                    out[static_cast<long long>(p.n_groups) * p.W] = q;
                }
            }
            const int d = t - q;
            const uint32_t ad = static_cast<uint32_t>(d < 0 ? -d : d);
            const uint32_t st = __reduce_add_sync(mask, static_cast<uint32_t>(t));
            const uint32_t sq = __reduce_add_sync(mask, static_cast<uint32_t>(q));
            const uint32_t sa = __reduce_add_sync(mask, ad);
            unsigned long long ss;
            if constexpr (kWide) {
                const unsigned long long d2 = static_cast<unsigned long long>(ad) * ad;       // < 2^53
                const uint32_t l0 = __reduce_add_sync(mask, static_cast<uint32_t>(d2 & 0x1fffffull));
                const uint32_t l1 = __reduce_add_sync(mask, static_cast<uint32_t>((d2 >> 21) & 0x1fffffull));
                const uint32_t l2 = __reduce_add_sync(mask, static_cast<uint32_t>(d2 >> 42));
                ss = static_cast<unsigned long long>(l0) + (static_cast<unsigned long long>(l1) << 21) +
                     (static_cast<unsigned long long>(l2) << 42);
            } else {
                ss = __reduce_add_sync(mask, ad * ad);
            }
            if (leader) {
                const int j = (g * p.n_regions + static_cast<int>(key)) * kSums;
                add_wide(s_lo + j, s_hi + j, st);
                add_wide(s_lo + j + 1, s_hi + j + 1, sq);
                add_wide(s_lo + j + 2, s_hi + j + 2, sa);
                add_wide(s_lo + j + 3, s_hi + j + 3, ss);
            }
        }
    }
    __syncthreads();
    unsigned long long* out = p.sums + vol * p.n_groups * p.n_regions * kStStats;
    for (int i = threadIdx.x; i < p.n_groups * p.n_regions * kStStats; i += kStThreads) {
        const int gr = i / kStStats, s = i - gr * kStStats;
        const unsigned long long v = s == 0 ? s_cnt[gr % p.n_regions]
                                            : (static_cast<unsigned long long>(s_hi[gr * kSums + s - 1]) << 32) |
                                                  s_lo[gr * kSums + s - 1];
        if (v != 0ull) atomicAdd(out + i, v);
    }
}

}  // namespace octm

// ----------------------------------------------------------------------------------- C ABI
extern "C" int octm_sector_thickness_i32(const int32_t* bnd_true, const int32_t* bnd_pred, int64_t n_items,
                                         int num_classes, int H, int W, int items_per_volume, const uint8_t* region,
                                         int n_regions, const int32_t* groups, int n_groups, int64_t* sums,
                                         int32_t* thick, void* stream) {
    if (n_items < 0 || H < 1 || W < 1) return octm::fail(OCTM_ERR_INVALID, "bad shape: n_items %lld, H %d, W %d",
                                                         static_cast<long long>(n_items), H, W);
    if (num_classes < 2 || num_classes > OCTM_MAX_CLASSES)
        return octm::fail(OCTM_ERR_INVALID, "num_classes %d outside [2, %d]", num_classes, OCTM_MAX_CLASSES);
    if (items_per_volume < 1 || n_items % items_per_volume != 0)
        return octm::fail(OCTM_ERR_INVALID, "items_per_volume %d must be >= 1 and divide n_items %lld", items_per_volume,
                          static_cast<long long>(n_items));
    if (n_regions < 1 || n_regions > octm::kStMaxRegions)
        return octm::fail(OCTM_ERR_INVALID, "n_regions %d outside [1, %d]", n_regions, octm::kStMaxRegions);
    if (n_groups < 1 || n_groups > octm::kStMaxGroups)
        return octm::fail(OCTM_ERR_INVALID, "n_groups %d outside [1, %d]", n_groups, octm::kStMaxGroups);
    if (groups == nullptr) return octm::fail(OCTM_ERR_INVALID, "null pointer: groups");
    octm::SectorParams p{};
    for (int g = 0; g < n_groups; ++g) {
        const int f = groups[2 * g], l = groups[2 * g + 1];
        if (f < 0 || f > l || l > num_classes - 1)
            return octm::fail(OCTM_ERR_INVALID, "groups[%d] = (%d, %d): need 0 <= first <= last <= %d", g, f, l,
                              num_classes - 1);
        p.first |= static_cast<unsigned long long>(f) << (4 * g);
        p.last |= static_cast<unsigned long long>(l) << (4 * g);
    }
    // the largest sum, sum (t - p)^2 over one volume, is below items_per_volume * W * H^2: exact in int64 and in float64
    const unsigned __int128 bound = static_cast<unsigned __int128>(items_per_volume) * static_cast<unsigned>(W) *
                                    static_cast<unsigned>(H) * static_cast<unsigned>(H);
    if (bound >= (static_cast<unsigned __int128>(1) << 53))
        return octm::fail(OCTM_ERR_INVALID, "items_per_volume * W * H^2 = %d * %d * %d^2 reaches 2^53: the sums would "
                          "not be exact", items_per_volume, W, H);
    if (n_items == 0) return OCTM_OK;
    if (!bnd_true || !bnd_pred || !region || !sums) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    const long long n_vol = n_items / items_per_volume;
    if (n_vol > 65535) return octm::fail(OCTM_ERR_UNSUPPORTED, "%lld volumes: at most 65535 per call", n_vol);
    const long long ascans = static_cast<long long>(items_per_volume) * W;
    // enough CTAs to fill the device a few times over, each at most kStMaxChunk A-scans
    const long long want = std::max(1ll, (ascans * n_vol + 4ll * octm::sm_count() - 1) / (4ll * octm::sm_count()));
    const int chunk = static_cast<int>(std::min<long long>(octm::kStMaxChunk,
        (want + octm::kStThreads - 1) / octm::kStThreads * octm::kStThreads));
    const long long chunks = (ascans + chunk - 1) / chunk;
    if (chunks > 0x7fffffffll) return octm::fail(OCTM_ERR_UNSUPPORTED, "volume too large");
    p.bnd_true = bnd_true;
    p.bnd_pred = bnd_pred;
    p.region = region;
    p.sums = reinterpret_cast<unsigned long long*>(sums);
    p.thick = thick;
    p.ascans = ascans;
    p.items_per_volume = items_per_volume;
    p.K = num_classes;
    p.H = H;
    p.W = W;
    p.n_regions = n_regions;
    p.n_groups = n_groups;
    p.chunk = chunk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t bytes = static_cast<size_t>(n_vol) * n_groups * n_regions * octm::kStStats * sizeof(int64_t);
    if (cudaMemsetAsync(sums, 0, bytes, st) != cudaSuccess) {
        cudaGetLastError();
        return octm::fail(OCTM_ERR_LAUNCH, "cudaMemsetAsync(sums) failed");
    }
    const dim3 grid(static_cast<unsigned>(chunks), static_cast<unsigned>(n_vol));
    if (H > 8192) {
        OCTM_TIMED("sector_thickness_kernel", st)
            octm::sector_thickness_kernel<true><<<grid, octm::kStThreads, 0, st>>>(p);
    } else {
        OCTM_TIMED("sector_thickness_kernel", st)
            octm::sector_thickness_kernel<false><<<grid, octm::kStThreads, 0, st>>>(p);
    }
    return octm::check_launch("sector_thickness_kernel");
}
