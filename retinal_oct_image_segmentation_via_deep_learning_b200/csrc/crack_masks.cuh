// Per-lane crack bitmasks of a label map (sm_100a): the crack arithmetic shared by the all-contour vertex emitter
// (contour_all.cu) and the surface Dice kernel (surface_dice.cu).
//
// A lane owns 16 columns [col0, col0 + 16) of image row y and forms, per class c, one 32-bit word:
//   bits  0..15  horizontal cracks (y, x) | (y, x + 1) with class c on exactly one side  (lattice row 2y,     x2 = 2x + 1)
//   bits 16..31  vertical cracks   (y, x) | (y + 1, x) with class c on exactly one side  (lattice row 2y + 1, x2 = 2x)
// bit b standing for column x = col0 + b.  The set bits over all rows are the all-contour vertex set of class c.
#pragma once

#include "common.cuh"

namespace octm {

constexpr uint32_t kFull = 0xffffffffu;

// 0x80 in every zero byte of z, 0 elsewhere (exact: no borrow between bytes)
__device__ __forceinline__ uint32_t zero_bytes(uint32_t z) {
    return ~(((z & 0x7f7f7f7fu) + 0x7f7f7f7fu) | z) & 0x80808080u;
}

// the four byte flags of zero_bytes -> bits 0..3 (byte b -> bit b)
__device__ __forceinline__ uint32_t byte_bits(uint32_t m) {
    return (m * 0x00204081u) >> 28;
}

// bit b set where label byte b of a equals label byte b of b_ (16 labels)
__device__ __forceinline__ uint32_t eq16(const uint4& a, const uint4& b_) {
    return byte_bits(zero_bytes(a.x ^ b_.x)) | byte_bits(zero_bytes(a.y ^ b_.y)) << 4 |
           byte_bits(zero_bytes(a.z ^ b_.z)) << 8 | byte_bits(zero_bytes(a.w ^ b_.w)) << 12;
}

// bit b set where label byte b of a equals the byte replicated in cc
__device__ __forceinline__ uint32_t eq16(const uint4& a, uint32_t cc) {
    return byte_bits(zero_bytes(a.x ^ cc)) | byte_bits(zero_bytes(a.y ^ cc)) << 4 |
           byte_bits(zero_bytes(a.z ^ cc)) << 8 | byte_bits(zero_bytes(a.w ^ cc)) << 12;
}

// labels [col0, col0 + 16) of one row; columns >= W read as 0 (the validity masks drop them)
template <bool VEC>
__device__ __forceinline__ uint4 load16(const uint8_t* row, int col0, int W) {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (col0 >= W) return v;
    if (VEC) return __ldg(reinterpret_cast<const uint4*>(row + col0));
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int b = 0; b < 16; ++b)
        if (col0 + b < W) w[b >> 2] |= static_cast<uint32_t>(__ldg(row + col0 + b)) << (8 * (b & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// Crack masks of the 16 columns [col0, col0 + 16) a lane owns in rows ra (= y) and rb (= y + 1, null on the last row):
// m[c] bits 0..15 = horizontal cracks (x, x + 1) with class c on one side, bits 16..31 = vertical cracks (y, x) | (y + 1, x).
// Returns false (warp-uniform, m untouched) when no lane of the warp has a crack.
template <bool VEC>
__device__ __forceinline__ bool crack_masks(const uint8_t* ra, const uint8_t* rb, int col0, int W, int K, int lane,
                                            uint32_t (&m)[OCTM_MAX_CLASSES]) {
    const uint4 a = load16<VEC>(ra, col0, W);
    const uint4 b = rb != nullptr ? load16<VEC>(rb, col0, W) : a;
    uint32_t nxt = __shfl_down_sync(kFull, a.x, 1);               // label of column col0 + 16 in byte 0
    if (lane == 31) nxt = col0 + 16 < W ? __ldg(ra + col0 + 16) : 0u;
    const uint4 a1 = make_uint4(__funnelshift_r(a.x, a.y, 8), __funnelshift_r(a.y, a.z, 8), __funnelshift_r(a.z, a.w, 8),
                                __funnelshift_r(a.w, nxt, 8));    // labels of columns x + 1
    const int nv = min(max(W - col0, 0), 16), nh = min(max(W - 1 - col0, 0), 16);
    const uint32_t dh = ~eq16(a, a1) & ((1u << nh) - 1u);
    const uint32_t dv = rb != nullptr ? ~eq16(a, b) & ((1u << nv) - 1u) : 0u;
    if (!__any_sync(kFull, (dh | dv) != 0u)) return false;
    const uint32_t nb = nxt & 0xffu;
#pragma unroll
    for (int c = 0; c < OCTM_MAX_CLASSES; ++c) {
        if (c >= K) break;
        const uint32_t cc = static_cast<uint32_t>(c) * 0x01010101u;
        const uint32_t ea = eq16(a, cc), eb = eq16(b, cc);
        const uint32_t ea1 = (ea >> 1) | (nb == static_cast<uint32_t>(c) ? 0x8000u : 0u);
        m[c] = ((ea | ea1) & dh) | (((ea | eb) & dv) << 16);
    }
    return true;
}

}  // namespace octm
