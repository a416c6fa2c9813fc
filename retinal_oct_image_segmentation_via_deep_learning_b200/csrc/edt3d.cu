// 3-D surface-distance metrics (BASELINE config 5): Hausdorff, HD95 and ASSD between the SURFACES of the
// class-c regions of two label volumes, by an exact separable squared-Euclidean distance transform.
//
// The reference's contour metrics (Metrics/Contour_based_metrics.py:5-56) are 2-D only; this is their
// 3-D counterpart with the customary definition (build-defined, SURVEY.md 8c item 4, oracle in
// oracle/surface3d_oracle.py):
//   surface(mask) = voxels of the mask with a 6-neighbour outside it (outside the volume counts as outside)
//                 = mask & ~scipy.ndimage.binary_erosion(mask)
//   direction 0: for every surface voxel of y_pred the squared distance to the nearest surface voxel of
//   y_true (unit spacing); direction 1 the other way round.  Per direction: count, max D2, the two order
//   statistics numpy's linear 95th percentile interpolates, sum of sqrt(D2) in float64 -- the same
//   integers / sums the 2-D kernels return, so derive.contour_metrics finishes both.
//
// Volume [D0][D1][D2], C-contiguous (D2 fastest).  Per (class, direction) unit:
//   pass 1 (along D2)  one thread per line: source-surface test from the labels (six neighbours), two
//                      sweeps -> g = distance along the line to the nearest surface voxel (uint16).
//   pass 2 (along D1)  one thread per line, adjacent threads = adjacent D2 (coalesced): Meijster lower
//                      envelope over (x - j)^2 + g(j)^2, the two stacks in local memory -> h2 (uint32).
//   pass 3 (along D0)  the same envelope over h2, evaluated only at the QUERY volume's surface voxels;
//                      the exact D2 values go into a histogram (shared-memory bins for small values,
//                      global atomics for the rest).
//   select             one CTA scans the histogram: count, max, order statistics, sum of count*sqrt(D2)
//                      in a fixed order (deterministic).
// octm_surface3d_spacing_u8 (end of the file) measures the same distances with a physical voxel spacing.
#include <cmath>
#include <cstdlib>
#include <type_traits>
#include <utility>

#include "common.cuh"

namespace octm {

constexpr uint16_t kInf16 = 0xffffu;
constexpr uint32_t kInf32 = 0xffffffffu;
constexpr int kMaxLine = 2048;           // longest D0 / D1 line (local-memory stacks of 2 x uint16 per element and thread)
constexpr int kSmemBins = 8192;          // squared distances below this are counted in shared memory

struct Edt3Params {
    const uint8_t* src;      // volume whose class surface is the source set
    const uint8_t* qry;      // volume whose class surface holds the query voxels
    int D0, D1, D2, cls;
    uint16_t* g;             // [D0][D1][D2]
    uint32_t* h2;            // [D0][D1][D2]
    uint32_t* hist;          // [nbins + 1]: bins, then the largest squared distance seen
    uint32_t nbins;
    const uint32_t* need;    // device word: 0 = the near-field path settled this unit, return at once (or null: always run)
};

__device__ __forceinline__ bool surface_at(const uint8_t* L, int D0, int D1, int D2, int i0, int i1, int i2, int cls) {
    const long long s1 = D2, s0 = static_cast<long long>(D1) * D2;
    const uint8_t* p = L + i0 * s0 + i1 * s1 + i2;
    if (*p != cls) return false;
    return i2 == 0 || p[-1] != cls || i2 == D2 - 1 || p[1] != cls || i1 == 0 || p[-s1] != cls || i1 == D1 - 1 || p[s1] != cls ||
           i0 == 0 || p[-s0] != cls || i0 == D0 - 1 || p[s0] != cls;
}

// ------------------------------------------------------------------------------------------ pass 1
__global__ void __launch_bounds__(128) edt3_pass1_kernel(const Edt3Params prm) {
    if (prm.need != nullptr && *prm.need == 0) return;
    const long long lines = static_cast<long long>(prm.D0) * prm.D1;
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2, cls = prm.cls;
    for (long long line = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; line < lines;
         line += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int i0 = static_cast<int>(line / D1), i1 = static_cast<int>(line % D1);
        const long long s0 = static_cast<long long>(D1) * D2;
        const uint8_t* c = prm.src + line * D2;
        const uint8_t* up = i0 > 0 ? c - s0 : nullptr;
        const uint8_t* dn = i0 < D0 - 1 ? c + s0 : nullptr;
        const uint8_t* lf = i1 > 0 ? c - D2 : nullptr;
        const uint8_t* rt = i1 < D1 - 1 ? c + D2 : nullptr;
        const bool border = !up || !dn || !lf || !rt;       // a missing neighbour line makes every mask voxel surface
        uint16_t* g = prm.g + line * D2;
        uint32_t dist = kInf16;
        int prev = -1, cur = c[0];
        for (int i2 = 0; i2 < D2; ++i2) {
            const int nxt = i2 + 1 < D2 ? c[i2 + 1] : -1;
            bool surf = false;
            if (cur == cls)
                surf = border || prev != cls || nxt != cls || up[i2] != cls || dn[i2] != cls || lf[i2] != cls || rt[i2] != cls;
            dist = surf ? 0u : (dist == kInf16 ? kInf16 : min(dist + 1u, 0xfffeu));
            g[i2] = static_cast<uint16_t>(dist);
            prev = cur;
            cur = nxt;
        }
        dist = kInf16;
        for (int i2 = D2 - 1; i2 >= 0; --i2) {
            const uint32_t f = g[i2];
            if (f == 0u) dist = 0u;
            else if (dist != kInf16) {
                dist = min(dist + 1u, 0xfffeu);
                if (dist < f) g[i2] = static_cast<uint16_t>(dist);
            }
        }
    }
}

// The same pass for D2 % 16 == 0 and 16-byte aligned volumes: the five label lines are read 16 voxels at a time
// (the byte-granular version is bound by the number of load instructions, not by bytes) and g leaves as two
// 16-byte stores per group; the backward sweep re-reads g group by group.
__device__ __forceinline__ uint32_t byte_of(const uint4& v, int i) {
    const uint32_t w = i < 8 ? (i < 4 ? v.x : v.y) : (i < 12 ? v.z : v.w);
    return (w >> ((i & 3) * 8)) & 0xffu;
}

__global__ void __launch_bounds__(128) edt3_pass1_vec_kernel(const Edt3Params prm) {
    if (prm.need != nullptr && *prm.need == 0) return;
    const long long lines = static_cast<long long>(prm.D0) * prm.D1;
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2;
    const uint32_t cls = static_cast<uint32_t>(prm.cls);
    const int groups = D2 / 16;
    for (long long line = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; line < lines;
         line += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int i0 = static_cast<int>(line / D1), i1 = static_cast<int>(line % D1);
        const long long s0 = static_cast<long long>(D1) * D2;
        const uint4* c = reinterpret_cast<const uint4*>(prm.src + line * D2);
        const bool border = i0 == 0 || i0 == D0 - 1 || i1 == 0 || i1 == D1 - 1;
        const uint4* up = border ? c : reinterpret_cast<const uint4*>(prm.src + line * D2 - s0);
        const uint4* dn = border ? c : reinterpret_cast<const uint4*>(prm.src + line * D2 + s0);
        const uint4* lf = border ? c : reinterpret_cast<const uint4*>(prm.src + line * D2 - D2);
        const uint4* rt = border ? c : reinterpret_cast<const uint4*>(prm.src + line * D2 + D2);
        uint4* g = reinterpret_cast<uint4*>(prm.g + line * D2);
        uint32_t dist = kInf16, prev = 0xffffffffu;
        uint4 cur = __ldg(c);
        for (int k = 0; k < groups; ++k) {
            const uint4 nxt = k + 1 < groups ? __ldg(c + k + 1) : make_uint4(~0u, ~0u, ~0u, ~0u);
            const uint4 u = __ldg(up + k), d = __ldg(dn + k), l = __ldg(lf + k), r = __ldg(rt + k);
            uint32_t out[8];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const uint32_t v = byte_of(cur, i);
                // past the end of the line: a value no class takes (the padding byte 0xff is class 255)
                const uint32_t nx = i < 15 ? byte_of(cur, i + 1) : (k + 1 < groups ? (nxt.x & 0xffu) : 0xffffffffu);
                bool surf = false;
                if (v == cls)
                    surf = border || prev != cls || nx != cls || byte_of(u, i) != cls || byte_of(d, i) != cls ||
                           byte_of(l, i) != cls || byte_of(r, i) != cls;
                dist = surf ? 0u : (dist == kInf16 ? kInf16 : min(dist + 1u, 0xfffeu));
                if (i & 1) out[i >> 1] |= dist << 16;
                else out[i >> 1] = dist;
                prev = v;
            }
            g[2 * k] = make_uint4(out[0], out[1], out[2], out[3]);
            g[2 * k + 1] = make_uint4(out[4], out[5], out[6], out[7]);
            cur = nxt;
        }
        dist = kInf16;
        for (int k = 2 * groups - 1; k >= 0; --k) {           // 8 values per 16-byte group, last to first
            uint4 w = g[k];
            uint32_t words[4] = {w.x, w.y, w.z, w.w};
            bool changed = false;
#pragma unroll
            for (int i = 7; i >= 0; --i) {
                const uint32_t f = (words[i >> 1] >> ((i & 1) * 16)) & 0xffffu;
                if (f == 0u) dist = 0u;
                else if (dist != kInf16) {
                    dist = min(dist + 1u, 0xfffeu);
                    if (dist < f) {
                        words[i >> 1] = (i & 1) ? ((words[i >> 1] & 0x0000ffffu) | (dist << 16)) : ((words[i >> 1] & 0xffff0000u) | dist);
                        changed = true;
                    }
                }
            }
            if (changed) g[k] = make_uint4(words[0], words[1], words[2], words[3]);
        }
    }
}

// ------------------------------------------------------------------------------------------ envelope
// Lower envelope of the parabolas  x -> a (x - j)^2 + w(j)  over the finite sites j of one line
// (Meijster et al.).  s[k] = site of region k, t[k] = first x of region k.  Returns the top index q
// (-1: the line has no finite site).  T = long long with a = 1: exact integers (voxel units); T = double: a is the
// squared spacing of the line's axis and every value is computed as a * (x - j)^2 + w(j), the expression the passes
// report.
template <class W, class T = decltype(std::declval<W>()(0))>
__device__ __forceinline__ int build_envelope(int n, W weight, uint16_t* s, uint16_t* t, T a = T(1)) {
    int q = -1;
    T wtop = 0;                                   // weight, site and first x of the top region, kept in registers
    long long itop = 0, ttop = 0;
    auto f = [a](long long x, long long i, T wi) -> T { return a * static_cast<T>((x - i) * (x - i)) + wi; };
    for (int u = 0; u < n; ++u) {
        const T wu = weight(u);
        if (wu < 0) continue;                                   // infinite site
        while (q >= 0) {
            const T fi = f(ttop, itop, wtop);
            const T fu = f(ttop, u, wu);
            if (fi <= fu) break;
            --q;                                                // u is lower over the whole top region: pop it
            if (q >= 0) {
                itop = s[q];
                ttop = t[q];
                wtop = weight(static_cast<int>(itop));
            }
        }
        if (q < 0) {
            q = 0;
            s[0] = static_cast<uint16_t>(u);
            t[0] = 0;
            itop = u; ttop = 0; wtop = wu;
        } else {
            long long sep;
            if constexpr (std::is_integral<T>::value) {
                // Meijster: Sep(i, u) = (u^2 - i^2 + w(u) - w(i)) div (2 (u - i)); u takes over from x = Sep + 1
                const long long num = static_cast<long long>(u) * u - itop * itop + wu - wtop;
                const long long den = 2 * (u - itop);
                sep = num >= 0 ? num / den : -((-num + den - 1) / den);       // floor division
            } else {
                // the rounded crossing of the two parabolas, then moved to the last x at which the top site's value is
                // still <= u's as f evaluates them (at ttop it is: the loop above stopped there), so that every region
                // holds the site of least reported value
                const double xc = ((wu - wtop) / a + static_cast<double>(static_cast<long long>(u) * u - itop * itop)) /
                                  (2.0 * static_cast<double>(u - itop));
                sep = xc >= n ? n - 1 : (xc <= ttop ? ttop : static_cast<long long>(floor(xc)));
                while (sep + 1 < n && f(sep + 1, itop, wtop) <= f(sep + 1, u, wu)) ++sep;
                while (sep > ttop && f(sep, itop, wtop) > f(sep, u, wu)) --sep;
            }
            const long long w = sep + 1;
            if (w < n) {
                ++q;
                s[q] = static_cast<uint16_t>(u);
                t[q] = static_cast<uint16_t>(w < 0 ? 0 : w);
                itop = u; ttop = w < 0 ? 0 : w; wtop = wu;
            }
        }
    }
    return q;
}

// ------------------------------------------------------------------------------------------ pass 2
__global__ void __launch_bounds__(128) edt3_pass2_kernel(const Edt3Params prm) {
    if (prm.need != nullptr && *prm.need == 0) return;
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2;
    const long long lines = static_cast<long long>(D0) * D2;
    uint16_t s[kMaxLine], t[kMaxLine];
    for (long long line = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; line < lines;
         line += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int i0 = static_cast<int>(line / D2), i2 = static_cast<int>(line % D2);
        const uint16_t* g = prm.g + static_cast<long long>(i0) * D1 * D2 + i2;       // element j at g[j * D2]
        uint32_t* h = prm.h2 + static_cast<long long>(i0) * D1 * D2 + i2;
        auto weight = [&](int j) -> long long {
            const uint32_t v = g[static_cast<long long>(j) * D2];
            return v == kInf16 ? -1ll : static_cast<long long>(v) * v;
        };
        int q = build_envelope(D1, weight, s, t);
        if (q < 0) {
            for (int x = 0; x < D1; ++x) h[static_cast<long long>(x) * D2] = kInf32;
            continue;
        }
        long long i = s[q], wi = weight(static_cast<int>(i));
        int tq = t[q];
        for (int x = D1 - 1; x >= 0; --x) {
            h[static_cast<long long>(x) * D2] = static_cast<uint32_t>((x - i) * (x - i) + wi);
            if (x == tq && q > 0) {
                --q;
                i = s[q];
                tq = t[q];
                wi = weight(static_cast<int>(i));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ pass 3
__global__ void __launch_bounds__(128) edt3_pass3_kernel(const Edt3Params prm) {
    __shared__ uint32_t s_hist[kSmemBins];
    if (prm.need != nullptr && *prm.need == 0) return;
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2, cls = prm.cls;
    const long long plane = static_cast<long long>(D1) * D2;
    for (int i = threadIdx.x; i < kSmemBins; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    uint16_t s[kMaxLine], t[kMaxLine];
    uint32_t big = 0;                                   // largest squared distance this thread sent to the global bins
    for (long long line = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; line < plane;
         line += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int i1 = static_cast<int>(line / D2), i2 = static_cast<int>(line % D2);
        const uint32_t* h = prm.h2 + line;                                          // element j at h[j * plane]
        auto weight = [&](int j) -> long long {
            const uint32_t v = h[static_cast<long long>(j) * plane];
            return v == kInf32 ? -1ll : static_cast<long long>(v);
        };
        int q = build_envelope(D0, weight, s, t);
        if (q < 0) continue;                                                        // no source surface at all
        long long i = s[q], wi = weight(static_cast<int>(i));
        int tq = t[q];
        for (int x = D0 - 1; x >= 0; --x) {
            if (surface_at(prm.qry, D0, D1, D2, x, i1, i2, cls)) {
                const uint32_t d2 = static_cast<uint32_t>((x - i) * (x - i) + wi);
                if (d2 < static_cast<uint32_t>(kSmemBins)) atomicAdd(&s_hist[d2], 1u);
                else {
                    atomicAdd(&prm.hist[min(d2, prm.nbins - 1)], 1u);
                    big = max(big, min(d2, prm.nbins - 1));
                }
            }
            if (x == tq && q > 0) {
                --q;
                i = s[q];
                tq = t[q];
                wi = weight(static_cast<int>(i));
            }
        }
    }
    __syncthreads();
    uint32_t top = 0;                                   // largest non-empty shared bin of this CTA
    for (int i = threadIdx.x; i < kSmemBins; i += blockDim.x) {
        const uint32_t c = s_hist[i];
        if (c && static_cast<uint32_t>(i) < prm.nbins) {
            atomicAdd(&prm.hist[i], c);
            top = i;
        }
    }
    top = max(top, big);
    top = __reduce_max_sync(0xffffffffu, top);
    if ((threadIdx.x & 31) == 0 && top) atomicMax(&prm.hist[prm.nbins], top);      // slot [nbins]: upper bound of the scan
}


// ================================================================================================ near-field path
// Surfaces of the same class in a prediction and its ground truth are a few voxels apart.  Distances below a cap
// (R + 1)^2 are exact under a CAPPED separable transform whose every pass looks only R voxels to either side:
//     G2(i2)  = min(CAP, g^2),                     g = distance along D2 to the nearest source surface voxel (<= R, else capped)
//     H2(i1)  = min(CAP, min_{|k| <= R} k^2 + G2(i1 + k))
//     D2(i0)  = min(CAP, min_{|k| <= R} k^2 + H2(i0 + k))        CAP = (R + 1)^2 <= 255
// Claim: D2 = min(CAP, true squared distance).  A source voxel at offset (a, b, c) with a^2 + b^2 + c^2 < CAP has
// |a|, |b|, |c| <= R, so it lies inside all three windows and none of its partial sums is capped; conversely every
// value below CAP that a pass produces is the squared distance to a real source voxel.  So whenever EVERY query voxel
// of a unit ends below CAP the unit's histogram is exact; otherwise a device flag is raised and the general (Meijster)
// kernels below redo the unit -- they return at once when the flag is clear.
// Planes are one BYTE per voxel, surfaces one BIT per voxel; the windowed minima run two voxels per instruction
// (VIADDMNMX.U16x2); pass 3 touches only the 16-row tiles that hold a query voxel.  No stacks, no local memory.
constexpr int kNearR = 10;
constexpr int kNearCap = (kNearR + 1) * (kNearR + 1);          // 121
constexpr int kNearTile = 16;                                  // output rows per thread in the windowed passes

struct NearParams {
    const uint8_t* vol;      // label volume
    int D0, D1, D2, cls;
    uint16_t* mask;          // [D0][D1][D2 / 16] surface bits of (vol == cls), bit j = voxel 16 g + j
    uint8_t* g2;             // [D0][D1][D2]
    uint8_t* h2;             // [D0][D1][D2]
    const uint16_t* qmask;   // query volume's surface bits
    uint32_t* hist;          // [nbins + 1]
    uint32_t nbins;
    uint32_t* overflow;      // device word: a query voxel at or beyond the cap
};

// 16 label bytes -> 16-bit mask of (byte == cls)
__device__ __forceinline__ uint32_t eq_mask16(const uint4& v, uint32_t c4) {
    auto nib = [&](uint32_t w) -> uint32_t {
        const uint32_t x = w ^ c4;
        const uint32_t z = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;      // exact zero-byte test
        return (((z >> 7) * 0x01020408u) >> 24) & 0xfu;
    };
    return nib(v.x) | (nib(v.y) << 4) | (nib(v.z) << 8) | (nib(v.w) << 12);
}

// surface bits of one class: thread = one group of 16 voxels along D2
__global__ void __launch_bounds__(256) near_surface_kernel(const NearParams prm) {
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2, G = D2 >> 4;
    const long long groups = static_cast<long long>(D0) * D1 * G;
    const uint32_t c4 = 0x01010101u * static_cast<uint32_t>(prm.cls);
    for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < groups;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int gk = static_cast<int>(t % G);
        const long long line = t / G;
        const int i1 = static_cast<int>(line % D1), i0 = static_cast<int>(line / D1);
        const uint8_t* c = prm.vol + line * D2 + gk * 16;
        const long long s0 = static_cast<long long>(D1) * D2;
        const uint32_t e = eq_mask16(__ldg(reinterpret_cast<const uint4*>(c)), c4);
        uint32_t inner = 0;                               // voxels whose six neighbours are all in the mask
        if (e != 0 && i0 > 0 && i0 < D0 - 1 && i1 > 0 && i1 < D1 - 1) {
            const uint32_t up = eq_mask16(__ldg(reinterpret_cast<const uint4*>(c - s0)), c4);
            const uint32_t dn = eq_mask16(__ldg(reinterpret_cast<const uint4*>(c + s0)), c4);
            const uint32_t lf = eq_mask16(__ldg(reinterpret_cast<const uint4*>(c - D2)), c4);
            const uint32_t rt = eq_mask16(__ldg(reinterpret_cast<const uint4*>(c + D2)), c4);
            const uint32_t pv = gk > 0 && c[-1] == prm.cls ? 1u : 0u, nx = gk < G - 1 && c[16] == prm.cls ? 1u : 0u;
            inner = up & dn & lf & rt & ((e << 1) | pv) & ((e >> 1) | (nx << 15));
        }
        prm.mask[t] = static_cast<uint16_t>(e & ~inner);
    }
}

// pass 1 from the bits: G2 of one group of 16 voxels from its own and its two neighbours' surface bits
__global__ void __launch_bounds__(256) near_pass1_kernel(const NearParams prm) {
    const int D2 = prm.D2, G = D2 >> 4;
    const long long groups = static_cast<long long>(prm.D0) * prm.D1 * G;
    for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < groups;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int gk = static_cast<int>(t % G);
        const unsigned long long ml = gk > 0 ? prm.mask[t - 1] : 0u, mc = prm.mask[t], mr = gk < G - 1 ? prm.mask[t + 1] : 0u;
        const unsigned long long w = ml | (mc << 16) | (mr << 32);       // bit 16 + j = voxel j of this group
        uint32_t out[4];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int p = 16 + j;
            const uint32_t right = static_cast<uint32_t>(w >> p) & ((2u << kNearR) - 1u);            // bit d: a surface voxel d to the right
            const uint32_t left = __brev(static_cast<uint32_t>(w >> (p - kNearR))) >> (31 - kNearR);   // bit d: d to the left
            const uint32_t both = right | left;
            const uint32_t g = both ? static_cast<uint32_t>(__ffs(both) - 1) : static_cast<uint32_t>(kNearR + 1);
            const uint32_t v = g * g;                                    // (R + 1)^2 = the cap
            if ((j & 3) == 0) out[j >> 2] = v;
            else out[j >> 2] |= v << ((j & 3) * 8);
        }
        reinterpret_cast<uint4*>(prm.g2)[t] = make_uint4(out[0], out[1], out[2], out[3]);
    }
}

// windowed minimum along one axis for 4 adjacent voxels x kNearTile rows: rows[] hold kNearTile + 2 R input words
// (4 bytes each) unpacked to two u16x2 registers; out row o = min(CAP, min_k k^2 + row[o + R + k])
struct NearRows {
    uint32_t lo[kNearTile + 2 * kNearR], hi[kNearTile + 2 * kNearR];
};
__device__ __forceinline__ void near_unpack(NearRows& r, int idx, uint32_t w) {
    r.lo[idx] = __byte_perm(w, 0, 0x4140);       // bytes 0, 1 -> halves
    r.hi[idx] = __byte_perm(w, 0, 0x4342);       // bytes 2, 3
}
__device__ __forceinline__ void near_window(const NearRows& r, int o, uint32_t& lo, uint32_t& hi) {
    lo = hi = static_cast<uint32_t>(kNearCap) * 0x00010001u;
#pragma unroll
    for (int k = -kNearR; k <= kNearR; ++k) {
        const uint32_t k2 = static_cast<uint32_t>(k * k) * 0x00010001u;
        lo = __viaddmin_u16x2(r.lo[o + kNearR + k], k2, lo);
        hi = __viaddmin_u16x2(r.hi[o + kNearR + k], k2, hi);
    }
}

// pass 2 (along D1): thread = (i0, tile of kNearTile rows of D1, 4 adjacent voxels of D2); a warp covers 128 voxels
__global__ void __launch_bounds__(128) near_pass2_kernel(const NearParams prm) {
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2, Q = D2 >> 2;
    const int tiles = (D1 + kNearTile - 1) / kNearTile;
    const long long total = static_cast<long long>(D0) * tiles * Q;
    const uint32_t capw = static_cast<uint32_t>(kNearCap) * 0x01010101u;
    for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int q = static_cast<int>(t % Q);
        const int tile = static_cast<int>((t / Q) % tiles), i0 = static_cast<int>(t / (static_cast<long long>(Q) * tiles));
        const int base = tile * kNearTile;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(prm.g2) + (static_cast<long long>(i0) * D1) * Q + q;
        NearRows r;
#pragma unroll
        for (int j = 0; j < kNearTile + 2 * kNearR; ++j) {
            const int i1 = base - kNearR + j;
            near_unpack(r, j, i1 >= 0 && i1 < D1 ? __ldg(src + static_cast<long long>(i1) * Q) : capw);
        }
        uint32_t* dst = reinterpret_cast<uint32_t*>(prm.h2) + (static_cast<long long>(i0) * D1) * Q + q;
#pragma unroll
        for (int o = 0; o < kNearTile; ++o) {
            if (base + o < D1) {
                uint32_t lo, hi;
                near_window(r, o, lo, hi);
                dst[static_cast<long long>(base + o) * Q] = __byte_perm(lo, hi, 0x6420);
            }
        }
    }
}

// pass 3 (along D0) at the query surface voxels + histogram: thread = (tile of kNearTile rows of D0, i1, 4 voxels)
__global__ void __launch_bounds__(128) near_pass3_kernel(const NearParams prm) {
    __shared__ uint32_t s_hist[kNearCap + 1];
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2, Q = D2 >> 2, G = D2 >> 4;
    const int tiles = (D0 + kNearTile - 1) / kNearTile;
    const long long plane_q = static_cast<long long>(D1) * Q, plane_g = static_cast<long long>(D1) * G;
    const long long total = static_cast<long long>(tiles) * plane_q;
    const uint32_t capw = static_cast<uint32_t>(kNearCap) * 0x01010101u;
    for (int i = threadIdx.x; i <= kNearCap; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long col = t % plane_q;                 // (i1, q)
        const int tile = static_cast<int>(t / plane_q), base = tile * kNearTile;
        const int q = static_cast<int>(col % Q);
        const long long gcol = (col / Q) * G + (q >> 2);   // (i1, group)
        const int sh = (q & 3) * 4;
        // the query bits of this thread's kNearTile x 4 voxels
        uint32_t bits[kNearTile / 8] = {};
        uint32_t any = 0;
#pragma unroll
        for (int o = 0; o < kNearTile; ++o) {
            const uint32_t nibble = base + o < D0 ? (static_cast<uint32_t>(__ldg(prm.qmask + (base + o) * plane_g + gcol)) >> sh) & 0xfu : 0u;
            bits[o >> 3] |= nibble << ((o & 7) * 4);
            any |= nibble;
        }
        if (any == 0) continue;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(prm.h2) + col;
        NearRows r;
#pragma unroll
        for (int j = 0; j < kNearTile + 2 * kNearR; ++j) {
            const int i0 = base - kNearR + j;
            near_unpack(r, j, i0 >= 0 && i0 < D0 ? __ldg(src + static_cast<long long>(i0) * plane_q) : capw);
        }
#pragma unroll
        for (int o = 0; o < kNearTile; ++o) {
            const uint32_t nibble = (bits[o >> 3] >> ((o & 7) * 4)) & 0xfu;
            if (nibble) {
                uint32_t lo, hi;
                near_window(r, o, lo, hi);
                const uint32_t v[4] = {lo & 0xffffu, lo >> 16, hi & 0xffffu, hi >> 16};
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if ((nibble >> j) & 1u) atomicAdd(&s_hist[v[j]], 1u);
            }
        }
    }
    __syncthreads();
    uint32_t top = 0;
    for (int i = threadIdx.x; i <= kNearCap; i += blockDim.x) {
        const uint32_t c = s_hist[i];
        if (c) {
            if (i == kNearCap) atomicOr(prm.overflow, 1u);
            else if (static_cast<uint32_t>(i) < prm.nbins) {
                atomicAdd(&prm.hist[i], c);
                top = i;
            }
        }
    }
    top = __reduce_max_sync(0xffffffffu, top);
    if ((threadIdx.x & 31) == 0 && top) atomicMax(&prm.hist[prm.nbins], top);
}

// the general kernels only run for a unit whose near-field attempt overflowed: clear its partial histogram
__global__ void __launch_bounds__(256) near_reset_kernel(uint32_t* hist, uint32_t n, const uint32_t* overflow) {
    if (*overflow == 0) return;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) hist[i] = 0;
}

// query-surface count when the source surface is empty is not needed: the metrics are undefined then.
// ------------------------------------------------------------------------------------------ select
struct Sel3Params {
    const uint32_t* hist;
    uint32_t nbins;
    uint32_t* n_pts;      // [1]
    uint32_t* max_sq;     // [1]
    uint32_t* p95_sq;     // [2]
    double* sum_dist;     // [1]
};

__global__ void __launch_bounds__(1024) edt3_select_kernel(const Sel3Params prm) {
    __shared__ unsigned long long s_scan[33];
    __shared__ double s_dsum[32];
    __shared__ uint32_t s_max[32];
    __shared__ uint32_t s_sel[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t n = min(prm.nbins, prm.hist[prm.nbins] + 1u);      // bins above the largest distance seen are empty
    const uint32_t chunk = (n + 1023u) / 1024u;
    const uint32_t b = min(n, tid * chunk), e = min(n, b + chunk);
    unsigned long long cnt = 0;
    uint32_t vmax = 0;
    double ds = 0.0;
    for (uint32_t v = b; v < e; ++v) {
        const uint32_t c = prm.hist[v];
        if (c) {
            cnt += c;
            vmax = v;
            ds = __dadd_rn(ds, __dmul_rn(static_cast<double>(c), sqrt(static_cast<double>(v))));
        }
    }
    unsigned long long total;
    const unsigned long long before = block_excl_scan_sum<unsigned long long>(cnt, s_scan, total);
    // fixed-order float64 sum: lanes tree, then warps in order
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ds = __dadd_rn(ds, __shfl_xor_sync(0xffffffffu, ds, o));
    vmax = __reduce_max_sync(0xffffffffu, vmax);
    if (lane == 0) { s_dsum[warp] = ds; s_max[warp] = vmax; }
    if (tid < 2) s_sel[tid] = 0;
    __syncthreads();
    if (total > 0) {
        // numpy linear percentile: virtual index (m - 1) * 0.95, neighbours floor and floor + 1
        const double pos = __dmul_rn(static_cast<double>(total - 1), 0.95);
        const unsigned long long k_lo = static_cast<unsigned long long>(floor(pos));
        const unsigned long long k_hi = k_lo + 1 < total ? k_lo + 1 : k_lo;
        unsigned long long run = before;
        for (uint32_t v = b; v < e; ++v) {
            const uint32_t c = prm.hist[v];
            if (c) {
                if (run <= k_lo && k_lo < run + c) s_sel[0] = v;
                if (run <= k_hi && k_hi < run + c) s_sel[1] = v;
                run += c;
            }
        }
    }
    __syncthreads();
    if (tid == 0) {
        double sum = 0.0;
        uint32_t m = 0;
        for (int w = 0; w < 32; ++w) { sum = __dadd_rn(sum, s_dsum[w]); m = max(m, s_max[w]); }
        prm.n_pts[0] = static_cast<uint32_t>(total > 0xffffffffull ? 0xffffffffull : total);
        prm.max_sq[0] = m;
        prm.p95_sq[0] = s_sel[0];
        prm.p95_sq[1] = s_sel[1];
        prm.sum_dist[0] = sum;
    }
}

// ================================================================================================ physical spacing
// octm_surface3d_spacing_u8: the same surfaces and directions, distances in the units of a voxel spacing (s0, s1, s2).
// With w_i = s_i^2 the squared distance to a source voxel at offset (a, b, c) is  d2 = w0 a^2 + (w1 b^2 + w2 c^2),
// evaluated in float64 in exactly that order: pass 2 forms w1 b^2 + w2 g^2, pass 3 adds w0 a^2.  Pass 1 (g, integer
// voxels along D2) does not depend on the weights and is the kernel above.  There is no integer histogram: pass 3
// stores the query voxels' d2 (their bit patterns: order-preserving for non-negative doubles) in one segment per CTA,
// the order statistics come from an 8-pass radix select over those bits, the sum of sqrt(d2) from per-CTA sums over a
// fixed set of lines added in a fixed order.  Everything is bit-reproducible.  The near-field path is not used (its
// byte planes hold integer squared distances).
constexpr int kW3Threads = 128;          // pass-3 CTA: one D0 line per thread, CTA b owns lines [128 b, 128 b + 128)
constexpr int kMaxTol = 4;
enum { kAccCount, kAccMax, kAccSurf, kAccWithin, kAccWords = kAccWithin + kMaxTol };

struct Edt3wParams {
    const uint8_t* qry;            // volume whose class surface holds the query voxels
    int D0, D1, D2, cls;
    const uint16_t* g;             // pass 1: [D0][D1][D2] distance along D2 in voxels
    double* h2;                    // [D0][D1][D2] w1 b^2 + w2 c^2 to the nearest source voxel of the i0 plane, -1: none
    double w0, w1, w2;
    double tau[kMaxTol];
    int ntau;
    unsigned long long* vals;      // [blocks][kW3Threads * D0] d2 bits of the query voxels of each pass-3 CTA
    uint32_t* seg_n;               // [blocks] values of each CTA
    double* seg_sum;               // [blocks] sum of sqrt(d2) of each CTA
    unsigned long long* acc;       // [kAccWords]: count, max d2 bits, query surface voxels, within each tolerance
};

__global__ void __launch_bounds__(128) edt3w_pass2_kernel(const Edt3wParams prm) {
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2;
    const double w1 = prm.w1, w2 = prm.w2;
    const long long lines = static_cast<long long>(D0) * D2;
    uint16_t s[kMaxLine], t[kMaxLine];
    for (long long line = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; line < lines;
         line += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int i0 = static_cast<int>(line / D2), i2 = static_cast<int>(line % D2);
        const uint16_t* g = prm.g + static_cast<long long>(i0) * D1 * D2 + i2;       // element j at g[j * D2]
        double* h = prm.h2 + static_cast<long long>(i0) * D1 * D2 + i2;
        auto weight = [&](int j) -> double {
            const uint32_t v = g[static_cast<long long>(j) * D2];
            return v == kInf16 ? -1.0 : w2 * static_cast<double>(v * v);
        };
        int q = build_envelope(D1, weight, s, t, w1);
        if (q < 0) {
            for (int x = 0; x < D1; ++x) h[static_cast<long long>(x) * D2] = -1.0;
            continue;
        }
        long long i = s[q];
        double wi = weight(static_cast<int>(i));
        int tq = t[q];
        for (int x = D1 - 1; x >= 0; --x) {
            h[static_cast<long long>(x) * D2] = w1 * static_cast<double>((x - i) * (x - i)) + wi;
            if (x == tq && q > 0) {
                --q;
                i = s[q];
                tq = t[q];
                wi = weight(static_cast<int>(i));
            }
        }
    }
}

__global__ void __launch_bounds__(kW3Threads) edt3w_pass3_kernel(const Edt3wParams prm) {
    __shared__ uint32_t s_n;
    __shared__ unsigned long long s_acc[kAccWords];
    __shared__ double s_sum[kW3Threads / 32];
    const int D0 = prm.D0, D1 = prm.D1, D2 = prm.D2, cls = prm.cls, tid = threadIdx.x;
    const long long plane = static_cast<long long>(D1) * D2;
    if (tid < kAccWords) s_acc[tid] = 0;
    if (tid == 0) s_n = 0;
    __syncthreads();
    unsigned long long* vals = prm.vals + static_cast<long long>(blockIdx.x) * kW3Threads * D0;
    const long long line = static_cast<long long>(blockIdx.x) * kW3Threads + tid;
    double sum = 0.0;
    unsigned long long mx = 0;
    uint32_t n = 0, nsurf = 0, within[kMaxTol] = {0, 0, 0, 0};
    if (line < plane) {
        uint16_t s[kMaxLine], t[kMaxLine];
        const int i1 = static_cast<int>(line / D2), i2 = static_cast<int>(line % D2);
        const double* h = prm.h2 + line;                                            // element j at h[j * plane]
        auto weight = [&](int j) -> double { return h[static_cast<long long>(j) * plane]; };
        const double w0 = prm.w0;
        int q = build_envelope(D0, weight, s, t, w0);                               // -1: no source surface at all
        long long i = q >= 0 ? s[q] : 0;
        double wi = q >= 0 ? weight(static_cast<int>(i)) : 0.0;
        int tq = q >= 0 ? t[q] : 0;
        for (int x = D0 - 1; x >= 0; --x) {
            if (surface_at(prm.qry, D0, D1, D2, x, i1, i2, cls)) {
                ++nsurf;                                                            // counted without a source too
                if (q >= 0) {
                    const double d2 = w0 * static_cast<double>((x - i) * (x - i)) + wi;
                    const double d = sqrt(d2);
                    sum = __dadd_rn(sum, d);
#pragma unroll
                    for (int j = 0; j < kMaxTol; ++j) within[j] += j < prm.ntau && d <= prm.tau[j] ? 1u : 0u;
                    const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(d2));
                    mx = max(mx, bits);
                    vals[atomicAdd(&s_n, 1u)] = bits;
                    ++n;
                }
            }
            if (x == tq && q > 0) {
                --q;
                i = s[q];
                tq = t[q];
                wi = weight(static_cast<int>(i));
            }
        }
    }
    // CTA totals: the float sum in a fixed order (lanes tree, then warps in order), integers by atomics
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    n = __reduce_add_sync(0xffffffffu, n);
    nsurf = __reduce_add_sync(0xffffffffu, nsurf);
#pragma unroll
    for (int j = 0; j < kMaxTol; ++j) within[j] = __reduce_add_sync(0xffffffffu, within[j]);
    if ((tid & 31) == 0) {
        s_sum[tid >> 5] = sum;
        atomicAdd(&s_acc[kAccCount], static_cast<unsigned long long>(n));
        atomicMax(&s_acc[kAccMax], mx);
        atomicAdd(&s_acc[kAccSurf], static_cast<unsigned long long>(nsurf));
        for (int j = 0; j < kMaxTol; ++j) atomicAdd(&s_acc[kAccWithin + j], static_cast<unsigned long long>(within[j]));
    }
    __syncthreads();
    if (tid == 0) {
        double cta = 0.0;
        for (int w = 0; w < kW3Threads / 32; ++w) cta = __dadd_rn(cta, s_sum[w]);
        prm.seg_sum[blockIdx.x] = cta;
        prm.seg_n[blockIdx.x] = s_n;
    }
    if (tid < kAccWords && s_acc[tid] != 0) {
        if (tid == kAccMax) atomicMax(&prm.acc[tid], s_acc[tid]);
        else atomicAdd(&prm.acc[tid], s_acc[tid]);
    }
}

struct Sel3wParams {
    const unsigned long long* vals;
    const uint32_t* seg_n;
    const double* seg_sum;
    const unsigned long long* acc;
    unsigned long long* hist;      // [8 passes][2 ranks][256]: digit counts of the values that share the rank's prefix
    long long seg_len;             // kW3Threads * D0
    int nseg, pass, ntau;
    uint32_t* n_pts;               // [1]
    double* max_sq;                // [1]
    double* p95_sq;                // [2]
    double* sum_dist;              // [1]
    uint32_t* n_surf;              // [1] or null
    uint32_t* n_within;            // [ntau]
};

// the two ranks numpy's linear 95th percentile interpolates between among m > 0 values (as edt3_select_kernel)
__device__ __forceinline__ void p95_ranks(unsigned long long m, unsigned long long& lo, unsigned long long& hi) {
    lo = static_cast<unsigned long long>(floor(__dmul_rn(static_cast<double>(m - 1), 0.95)));
    hi = lo + 1 < m ? lo + 1 : lo;
}

// One warp: the top 8 * passes bits of the value of rank k, from the digit counts of the first `passes` passes (h: this
// rank's counts of pass 0, 512 apart per pass).  Every lane returns the same prefix.
__device__ unsigned long long radix_prefix(const unsigned long long* h, int passes, unsigned long long k) {
    const int lane = threadIdx.x & 31;
    unsigned long long prefix = 0, rank = k;
    for (int p = 0; p < passes; ++p, h += 512) {
        unsigned long long c[8], tot = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { c[j] = h[lane * 8 + j]; tot += c[j]; }
        unsigned long long inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        const unsigned long long exc = inc - tot;
        const bool mine = exc <= rank && rank < inc;
        const int owner = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
        int d = 0;
        unsigned long long r = rank - exc;
        if (mine) {
            for (int j = 0; j < 8; ++j) {
                if (r < c[j]) { d = lane * 8 + j; break; }
                r -= c[j];
            }
        }
        prefix = (prefix << 8) | static_cast<unsigned long long>(__shfl_sync(0xffffffffu, d, owner));
        rank = __shfl_sync(0xffffffffu, r, owner);
    }
    return prefix;
}

// radix-select pass p: digit p (bits 63 - 8p .. 56 - 8p) of the values whose top 8p bits are the prefix of either rank
__global__ void __launch_bounds__(256) edt3w_radix_kernel(const Sel3wParams prm) {
    __shared__ unsigned long long s_hist[512];
    __shared__ unsigned long long s_prefix[2];
    const unsigned long long m = prm.acc[kAccCount];
    if (m == 0) return;
    const int p = prm.pass, tid = threadIdx.x;
    for (int i = tid; i < 512; i += blockDim.x) s_hist[i] = 0;
    if (tid < 32) {
        unsigned long long lo, hi;
        p95_ranks(m, lo, hi);
        const unsigned long long pl = radix_prefix(prm.hist, p, lo), ph = radix_prefix(prm.hist + 256, p, hi);
        if (tid == 0) { s_prefix[0] = pl; s_prefix[1] = ph; }
    }
    __syncthreads();
    const int shift = 56 - 8 * p;
    const unsigned long long pl = s_prefix[0], ph = s_prefix[1];
    for (int seg = blockIdx.x; seg < prm.nseg; seg += gridDim.x) {
        const uint32_t n = prm.seg_n[seg];
        const unsigned long long* v = prm.vals + seg * prm.seg_len;
        // most values share their top digits: the lanes of a warp that hit the same counter add to it once
        // (the loop bound is uniform over the CTA, so every warp is converged at the match)
        for (uint32_t base = 0; base < n; base += blockDim.x) {
            const uint32_t e = base + tid;
            uint32_t klo = 0xffffffffu, khi = 0xffffffffu;
            if (e < n) {
                const unsigned long long x = v[e];
                const unsigned long long top = p == 0 ? 0ull : x >> (shift + 8);
                const uint32_t d = static_cast<uint32_t>(x >> shift) & 0xffu;
                if (top == pl) klo = d;
                if (top == ph) khi = 256 + d;
            }
            const uint32_t mlo = __match_any_sync(0xffffffffu, klo), mhi = __match_any_sync(0xffffffffu, khi);
            if (klo != 0xffffffffu && (mlo & lanemask_lt()) == 0) atomicAdd(&s_hist[klo], static_cast<unsigned long long>(__popc(mlo)));
            if (khi != 0xffffffffu && (mhi & lanemask_lt()) == 0) atomicAdd(&s_hist[khi], static_cast<unsigned long long>(__popc(mhi)));
        }
    }
    __syncthreads();
    for (int i = tid; i < 512; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&prm.hist[p * 512 + i], s_hist[i]);
}

__global__ void __launch_bounds__(1024) edt3w_finish_kernel(const Sel3wParams prm) {
    __shared__ double s_dsum[32];
    __shared__ unsigned long long s_sel[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long m = prm.acc[kAccCount];
    // fixed-order float64 sum of the per-CTA sums: contiguous chunks per thread, lanes tree, warps in order
    const int chunk = (prm.nseg + 1023) / 1024;
    const int b = min(prm.nseg, tid * chunk), e = min(prm.nseg, b + chunk);
    double ds = 0.0;
    for (int v = b; v < e; ++v) ds = __dadd_rn(ds, prm.seg_sum[v]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ds = __dadd_rn(ds, __shfl_xor_sync(0xffffffffu, ds, o));
    if (lane == 0) s_dsum[warp] = ds;
    if (warp == 0) {
        unsigned long long lo = 0, hi = 0, vl = 0, vh = 0;
        if (m > 0) {
            p95_ranks(m, lo, hi);
            vl = radix_prefix(prm.hist, 8, lo);
            vh = radix_prefix(prm.hist + 256, 8, hi);
        }
        if (lane == 0) { s_sel[0] = vl; s_sel[1] = vh; }
    }
    __syncthreads();
    if (tid == 0) {
        double sum = 0.0;
        for (int w = 0; w < 32; ++w) sum = __dadd_rn(sum, s_dsum[w]);
        auto clamp32 = [](unsigned long long v) { return static_cast<uint32_t>(v > 0xffffffffull ? 0xffffffffull : v); };
        prm.n_pts[0] = clamp32(m);
        prm.max_sq[0] = __longlong_as_double(static_cast<long long>(prm.acc[kAccMax]));
        prm.p95_sq[0] = __longlong_as_double(static_cast<long long>(s_sel[0]));
        prm.p95_sq[1] = __longlong_as_double(static_cast<long long>(s_sel[1]));
        prm.sum_dist[0] = sum;
        if (prm.n_surf) prm.n_surf[0] = clamp32(prm.acc[kAccSurf]);
        for (int j = 0; j < prm.ntau; ++j) prm.n_within[j] = clamp32(prm.acc[kAccWithin + j]);
    }
}

}  // namespace octm

static uint32_t edt3_nbins(int D0, int D1, int D2) {
    const unsigned long long m = 1ull * (D0 - 1) * (D0 - 1) + 1ull * (D1 - 1) * (D1 - 1) + 1ull * (D2 - 1) * (D2 - 1) + 1ull;
    return static_cast<uint32_t>(m);
}

extern "C" size_t octm_surface3d_workspace_bytes(int D0, int D1, int D2) {
    if (D0 < 1 || D1 < 1 || D2 < 1) return 0;
    const size_t vox = static_cast<size_t>(D0) * D1 * D2;
    auto up = [](size_t v) { return (v + 255) & ~static_cast<size_t>(255); };
    // general path: g (uint16), h2 (uint32), histogram; near-field path: two surface bit masks and a flag of their own (its
    // byte planes live inside g: the general kernels only run after the near-field results of a unit are abandoned)
    return up(vox * 2) + up(vox * 4) + up((static_cast<size_t>(edt3_nbins(D0, D1, D2)) + 1) * 4) + 2 * up(vox / 16 * 2 + 2) + 256;
}

extern "C" int octm_surface3d_u8(const uint8_t* y_true, const uint8_t* y_pred, int D0, int D1, int D2, int num_classes,
                                 int unit_begin, int unit_end, uint32_t* n_pts, uint32_t* max_sq, uint32_t* p95_sq,
                                 double* sum_dist, void* workspace, size_t workspace_bytes, void* stream) {
    if (D0 < 1 || D1 < 1 || D2 < 1) return octm::fail(OCTM_ERR_INVALID, "bad volume shape");
    if (num_classes < 1 || num_classes > 256) return octm::fail(OCTM_ERR_INVALID, "num_classes outside [1, 256]");
    if (unit_begin < 0 || unit_end > 2 * num_classes || unit_begin > unit_end) return octm::fail(OCTM_ERR_INVALID, "bad unit range");
    if (D0 > octm::kMaxLine || D1 > octm::kMaxLine || D2 > 65534)
        return octm::fail(OCTM_ERR_UNSUPPORTED, "volume sides: D0, D1 <= %d and D2 <= 65534", octm::kMaxLine);
    const unsigned long long far2 = 1ull * (D0 - 1) * (D0 - 1) + 1ull * (D1 - 1) * (D1 - 1) + 1ull * (D2 - 1) * (D2 - 1);
    if (far2 >= (1ull << 28)) return octm::fail(OCTM_ERR_UNSUPPORTED, "squared diagonal %llu needs a histogram of more than 2^28 bins", far2);
    if (!y_true || !y_pred || !n_pts || !max_sq || !p95_sq || !sum_dist) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    if (workspace == nullptr || workspace_bytes < octm_surface3d_workspace_bytes(D0, D1, D2))
        return octm::fail(OCTM_ERR_WORKSPACE, "workspace too small: need %zu B", octm_surface3d_workspace_bytes(D0, D1, D2));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t vox = static_cast<size_t>(D0) * D1 * D2;
    auto up = [](size_t v) { return (v + 255) & ~static_cast<size_t>(255); };
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    uint16_t* g = reinterpret_cast<uint16_t*>(ws);
    uint32_t* h2 = reinterpret_cast<uint32_t*>(ws + up(vox * 2));
    uint32_t* hist = reinterpret_cast<uint32_t*>(ws + up(vox * 2) + up(vox * 4));
    const uint32_t nbins = edt3_nbins(D0, D1, D2);
    const int sms = octm::sm_count();
    // near-field path (see above): byte planes inside the general path's g region, bit masks and the flag after the histogram
    const bool near_ok = D2 % 16 == 0 && reinterpret_cast<uintptr_t>(y_true) % 16 == 0 &&
                         reinterpret_cast<uintptr_t>(y_pred) % 16 == 0;
    uint8_t* ng2 = reinterpret_cast<uint8_t*>(g);
    uint8_t* nh2 = ng2 + up(vox);
    const size_t mask_elems = vox / 16;
    uint8_t* tail = reinterpret_cast<uint8_t*>(hist) + up((static_cast<size_t>(edt3_nbins(D0, D1, D2)) + 1) * 4);
    uint16_t* mask_t = reinterpret_cast<uint16_t*>(tail);
    uint16_t* mask_p = reinterpret_cast<uint16_t*>(tail + up(mask_elems * 2 + 2));
    uint32_t* overflow = reinterpret_cast<uint32_t*>(tail + 2 * up(mask_elems * 2 + 2));
    int masks_of_class = -1;
    auto grid_for = [&](long long threads, int block) {
        long long b = (threads + block - 1) / block;
        const long long cap = static_cast<long long>(sms) * 32;
        return static_cast<unsigned>(b < cap ? b : cap);
    };
    // the Meijster kernels keep 2 x kMaxLine uint16 of stack per thread in local memory
    for (int unit = unit_begin; unit < unit_end; ++unit) {
        const int cls = unit >> 1, dir = unit & 1;
        // direction 0: queries = y_pred surface, sources = y_true surface (d1 of the reference); 1 swapped
        octm::Edt3Params p{dir == 0 ? y_true : y_pred, dir == 0 ? y_pred : y_true, D0, D1, D2, cls, g, h2, hist, nbins,
                           near_ok ? overflow : nullptr};
        if (cudaMemsetAsync(hist, 0, (static_cast<size_t>(nbins) + 1) * 4, st) != cudaSuccess)
            return octm::fail(OCTM_ERR_LAUNCH, "memset(hist) failed");
        if (near_ok) {
            if (cudaMemsetAsync(overflow, 0, 4, st) != cudaSuccess) return octm::fail(OCTM_ERR_LAUNCH, "memset failed");
            octm::NearParams np{nullptr, D0, D1, D2, cls, nullptr, ng2, nh2, nullptr, hist, nbins, overflow};
            if (masks_of_class != cls) {                 // surface bits of both volumes: shared by the class's two directions
                np.vol = y_true; np.mask = mask_t;
                OCTM_TIMED("near_surface_kernel", st) octm::near_surface_kernel<<<grid_for(static_cast<long long>(mask_elems), 256), 256, 0, st>>>(np);
                np.vol = y_pred; np.mask = mask_p;
                OCTM_TIMED("near_surface_kernel", st) octm::near_surface_kernel<<<grid_for(static_cast<long long>(mask_elems), 256), 256, 0, st>>>(np);
                if (int e = octm::check_launch("near_surface_kernel")) return e;
                masks_of_class = cls;
            }
            np.mask = dir == 0 ? mask_t : mask_p;        // sources
            np.qmask = dir == 0 ? mask_p : mask_t;       // queries
            OCTM_TIMED("near_pass1_kernel", st) octm::near_pass1_kernel<<<grid_for(static_cast<long long>(mask_elems), 256), 256, 0, st>>>(np);
            if (int e = octm::check_launch("near_pass1_kernel")) return e;
            const long long t2 = 1ll * D0 * ((D1 + octm::kNearTile - 1) / octm::kNearTile) * (D2 / 4);
            OCTM_TIMED("near_pass2_kernel", st) octm::near_pass2_kernel<<<grid_for(t2, 128), 128, 0, st>>>(np);
            if (int e = octm::check_launch("near_pass2_kernel")) return e;
            const long long t3 = 1ll * ((D0 + octm::kNearTile - 1) / octm::kNearTile) * D1 * (D2 / 4);
            OCTM_TIMED("near_pass3_kernel", st) octm::near_pass3_kernel<<<grid_for(t3, 128), 128, 0, st>>>(np);
            if (int e = octm::check_launch("near_pass3_kernel")) return e;
            // a query voxel at or beyond the cap: the general kernels below redo the unit from a clean histogram
            OCTM_TIMED("near_reset_kernel", st) octm::near_reset_kernel<<<static_cast<unsigned>(sms), 256, 0, st>>>(hist, nbins + 1, overflow);
            if (int e = octm::check_launch("near_reset_kernel")) return e;
        }
        auto blocks = [&](long long threads) {
            long long b = (threads + 127) / 128;
            const long long cap = static_cast<long long>(sms) * 16;
            return static_cast<unsigned>(b < cap ? b : cap);
        };
        if (D2 % 16 == 0 && reinterpret_cast<uintptr_t>(p.src) % 16 == 0)
            OCTM_TIMED("edt3_pass1_vec_kernel", st) octm::edt3_pass1_vec_kernel<<<blocks(1ll * D0 * D1), 128, 0, st>>>(p);
        else
            OCTM_TIMED("edt3_pass1_kernel", st) octm::edt3_pass1_kernel<<<blocks(1ll * D0 * D1), 128, 0, st>>>(p);
        if (int e = octm::check_launch("edt3_pass1_kernel")) return e;
        OCTM_TIMED("edt3_pass2_kernel", st) octm::edt3_pass2_kernel<<<blocks(1ll * D0 * D2), 128, 0, st>>>(p);
        if (int e = octm::check_launch("edt3_pass2_kernel")) return e;
        OCTM_TIMED("edt3_pass3_kernel", st) octm::edt3_pass3_kernel<<<blocks(1ll * D1 * D2), 128, 0, st>>>(p);
        if (int e = octm::check_launch("edt3_pass3_kernel")) return e;
        // n_pts keeps the 2-D layout [K][2] = (surface voxels of y_true, of y_pred): direction 0 queries y_pred's
        octm::Sel3Params sp{hist, nbins, n_pts + cls * 2 + (1 - dir), max_sq + unit, p95_sq + 2 * unit, sum_dist + unit};
        OCTM_TIMED("edt3_select_kernel", st) octm::edt3_select_kernel<<<1, 1024, 0, st>>>(sp);
        if (int e = octm::check_launch("edt3_select_kernel")) return e;
    }
    return OCTM_OK;
}

// physical-spacing workspace: g and then the pass-3 value segments (g is dead once pass 2 has run), h2 (float64), the
// per-CTA counts and sums of pass 3, the unit's totals and radix-select digit counts
namespace {
struct Edt3wLayout {
    size_t vals, h2, seg_n, seg_sum, acc, total;
    long long nseg;
};
Edt3wLayout edt3w_layout(int D0, int D1, int D2) {
    auto up = [](size_t v) { return (v + 255) & ~static_cast<size_t>(255); };
    Edt3wLayout L{};
    const size_t vox = static_cast<size_t>(D0) * D1 * D2;
    L.nseg = (static_cast<long long>(D1) * D2 + octm::kW3Threads - 1) / octm::kW3Threads;
    L.vals = 0;
    L.h2 = L.vals + up(static_cast<size_t>(L.nseg) * octm::kW3Threads * D0 * 8);
    L.seg_n = L.h2 + up(vox * 8);
    L.seg_sum = L.seg_n + up(static_cast<size_t>(L.nseg) * 4);
    L.acc = L.seg_sum + up(static_cast<size_t>(L.nseg) * 8);
    L.total = L.acc + up((octm::kAccWords + 8 * 512) * 8);
    return L;
}
}  // namespace

extern "C" size_t octm_surface3d_spacing_workspace_bytes(int D0, int D1, int D2) {
    if (D0 < 1 || D1 < 1 || D2 < 1) return 0;
    return edt3w_layout(D0, D1, D2).total;
}

extern "C" int octm_surface3d_spacing_u8(const uint8_t* y_true, const uint8_t* y_pred, int D0, int D1, int D2,
                                         int num_classes, int unit_begin, int unit_end, const double* spacing,
                                         const double* tolerances, int num_tolerances, uint32_t* n_pts, double* max_sq,
                                         double* p95_sq, double* sum_dist, uint32_t* n_surf, uint32_t* n_within,
                                         void* workspace, size_t workspace_bytes, void* stream) {
    if (D0 < 1 || D1 < 1 || D2 < 1) return octm::fail(OCTM_ERR_INVALID, "bad volume shape");
    if (num_classes < 1 || num_classes > 256) return octm::fail(OCTM_ERR_INVALID, "num_classes outside [1, 256]");
    if (unit_begin < 0 || unit_end > 2 * num_classes || unit_begin > unit_end) return octm::fail(OCTM_ERR_INVALID, "bad unit range");
    if (D0 > octm::kMaxLine || D1 > octm::kMaxLine || D2 > 65534)
        return octm::fail(OCTM_ERR_UNSUPPORTED, "volume sides: D0, D1 <= %d and D2 <= 65534", octm::kMaxLine);
    if (!y_true || !y_pred || !n_pts || !max_sq || !p95_sq || !sum_dist || !spacing) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    for (int a = 0; a < 3; ++a)
        if (!std::isfinite(spacing[a]) || !(spacing[a] > 0.0))
            return octm::fail(OCTM_ERR_INVALID, "spacing[%d] = %g: must be finite and > 0", a, spacing[a]);
    // the kernels work with w = spacing^2: it must be a normal double (no overflow to inf, no underflow to 0 or
    // subnormals), and so must the largest squared distance the volume can hold
    for (int a = 0; a < 3; ++a)
        if (!std::isnormal(spacing[a] * spacing[a]))
            return octm::fail(OCTM_ERR_INVALID, "spacing[%d] = %g: its square is not a normal double", a, spacing[a]);
    const double diag2 = spacing[0] * spacing[0] * (1.0 * (D0 - 1) * (D0 - 1)) + spacing[1] * spacing[1] * (1.0 * (D1 - 1) * (D1 - 1)) +
                         spacing[2] * spacing[2] * (1.0 * (D2 - 1) * (D2 - 1));
    if (!std::isfinite(diag2))
        return octm::fail(OCTM_ERR_INVALID, "spacing: the squared diagonal of the volume overflows a double");
    if (num_tolerances < 0 || num_tolerances > octm::kMaxTol)
        return octm::fail(OCTM_ERR_INVALID, "num_tolerances %d outside [0, %d]", num_tolerances, octm::kMaxTol);
    if (num_tolerances > 0 && (!tolerances || !n_surf || !n_within))
        return octm::fail(OCTM_ERR_INVALID, "null pointer: tolerances, n_surf and n_within are needed with tolerances");
    for (int j = 0; j < num_tolerances; ++j)
        if (!std::isfinite(tolerances[j]) || !(tolerances[j] >= 0.0))
            return octm::fail(OCTM_ERR_INVALID, "tolerances[%d] = %g: must be finite and >= 0", j, tolerances[j]);
    const Edt3wLayout L = edt3w_layout(D0, D1, D2);
    if (workspace == nullptr || workspace_bytes < L.total)
        return octm::fail(OCTM_ERR_WORKSPACE, "workspace too small: need %zu B", L.total);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    uint16_t* g = reinterpret_cast<uint16_t*>(ws + L.vals);
    unsigned long long* vals = reinterpret_cast<unsigned long long*>(ws + L.vals);
    double* h2 = reinterpret_cast<double*>(ws + L.h2);
    uint32_t* seg_n = reinterpret_cast<uint32_t*>(ws + L.seg_n);
    double* seg_sum = reinterpret_cast<double*>(ws + L.seg_sum);
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(ws + L.acc);
    unsigned long long* hist = acc + octm::kAccWords;
    const int sms = octm::sm_count();
    auto blocks = [&](long long threads, long long per_sm) {
        long long b = (threads + 127) / 128;
        const long long cap = static_cast<long long>(sms) * per_sm;
        return static_cast<unsigned>(b < cap ? b : cap);
    };
    octm::Edt3wParams wp{};
    wp.D0 = D0; wp.D1 = D1; wp.D2 = D2;
    wp.g = g; wp.h2 = h2;
    wp.w0 = spacing[0] * spacing[0];
    wp.w1 = spacing[1] * spacing[1];
    wp.w2 = spacing[2] * spacing[2];
    for (int j = 0; j < num_tolerances; ++j) wp.tau[j] = tolerances[j];
    wp.ntau = num_tolerances;
    wp.vals = vals; wp.seg_n = seg_n; wp.seg_sum = seg_sum; wp.acc = acc;
    for (int unit = unit_begin; unit < unit_end; ++unit) {
        const int cls = unit >> 1, dir = unit & 1;
        // direction 0: queries = y_pred surface, sources = y_true surface; 1 swapped (as octm_surface3d_u8)
        const uint8_t* src = dir == 0 ? y_true : y_pred;
        octm::Edt3Params p{src, nullptr, D0, D1, D2, cls, g, nullptr, nullptr, 0, nullptr};
        wp.qry = dir == 0 ? y_pred : y_true;
        wp.cls = cls;
        if (cudaMemsetAsync(acc, 0, (octm::kAccWords + 8 * 512) * 8, st) != cudaSuccess)
            return octm::fail(OCTM_ERR_LAUNCH, "memset(acc) failed");
        if (D2 % 16 == 0 && reinterpret_cast<uintptr_t>(src) % 16 == 0)
            OCTM_TIMED("edt3_pass1_vec_kernel", st) octm::edt3_pass1_vec_kernel<<<blocks(1ll * D0 * D1, 16), 128, 0, st>>>(p);
        else
            OCTM_TIMED("edt3_pass1_kernel", st) octm::edt3_pass1_kernel<<<blocks(1ll * D0 * D1, 16), 128, 0, st>>>(p);
        if (int e = octm::check_launch("edt3_pass1_kernel")) return e;
        OCTM_TIMED("edt3w_pass2_kernel", st) octm::edt3w_pass2_kernel<<<blocks(1ll * D0 * D2, 16), 128, 0, st>>>(wp);
        if (int e = octm::check_launch("edt3w_pass2_kernel")) return e;
        OCTM_TIMED("edt3w_pass3_kernel", st) octm::edt3w_pass3_kernel<<<static_cast<unsigned>(L.nseg), octm::kW3Threads, 0, st>>>(wp);
        if (int e = octm::check_launch("edt3w_pass3_kernel")) return e;
        // n_pts and n_surf keep the layout [K][2] = (y_true, y_pred): direction 0 queries y_pred's surface
        octm::Sel3wParams sp{vals, seg_n, seg_sum, acc, hist, 1ll * octm::kW3Threads * D0, static_cast<int>(L.nseg), 0,
                             num_tolerances, n_pts + cls * 2 + (1 - dir), max_sq + unit, p95_sq + 2 * unit, sum_dist + unit,
                             n_surf ? n_surf + cls * 2 + (1 - dir) : nullptr,
                             n_within ? n_within + unit * num_tolerances : nullptr};
        for (sp.pass = 0; sp.pass < 8; ++sp.pass) {
            OCTM_TIMED("edt3w_radix_kernel", st) octm::edt3w_radix_kernel<<<blocks(L.nseg * 128, 2), 256, 0, st>>>(sp);
            if (int e = octm::check_launch("edt3w_radix_kernel")) return e;
        }
        OCTM_TIMED("edt3w_finish_kernel", st) octm::edt3w_finish_kernel<<<1, 1024, 0, st>>>(sp);
        if (int e = octm::check_launch("edt3w_finish_kernel")) return e;
    }
    return OCTM_OK;
}
