// Fused label pass: confusion matrix (K1) + column scan (K2) + boundary error (K3) + contour
// seeds, in one read of the two uint8 label tensors.  sm_100a only.
//
// Replaces, for all classes at once, the per-class numpy passes of the reference:
//   Metrics/ConfusionMatrix_based_metrics.py:14-17,30-32,45-47,60-62   (sum-of-products counts)
//   Metrics/Region_based_metrics.py:13-15,28-30,43-45,58-60
//   Metrics/Biomarker_based_metrics.py:14-21                            (column sums, |dt|)
// plus the build-defined boundary positions b_k(x) = #{y : L[y][x] < k}  (SURVEY.md 8a-D).
//
// FAST KERNEL (W % 16 == 0, W <= 2048, H <= 4096, K <= 8)
//   * persistent CTAs, one B-scan at a time, one warp per strip of 128 columns for ALL rows of the
//     item.  Every warp owns a private shared-memory ring (S stages x 2 maps x R rows x 128 B) that it
//     fills itself with 2-D TMA tile copies (cp.async.bulk.tensor.2d -> UTMALDG, evict-first) completing
//     on its own mbarriers: no producer warp, no cross-warp wait inside an item.
//   * lane = 8 adjacent columns (one LDS.64 per map); lanes 0-15 take the even row of a row pair,
//     lanes 16-31 the odd row.  Column state therefore never crosses warps.
//   * column scan: labels of 4 pixels x 2 maps are interleaved into a PRMT selector; one PRMT against
//     an 8-entry byte LUT (immediate) yields the flags of a PAIR of thresholds; flags accumulate in
//     nibble counters (IMAD adds on the FMA pipe), flushed every 28 rows into byte counters, those every
//     504 rows (126 four-row groups) into uint16 column totals in shared memory.
//   * confusion matrix: joint code t*8+p per pixel.  A lane whose 16 pixel pairs share one code (the
//     common case in segmentation maps) extends a run counted in a register; runs reach the lane's
//     private uint16 histogram column when the code changes.  The rare mixed lanes are compacted
//     (ballot + popc) into a per-warp queue and drained 32 entries at a time, one entry per lane.
//   * contour seeds: classes are tracked per warp; lanes that meet a new class record its first raster
//     position with a shared-memory atomicMin.
//   * without the histogram (CONF = 0, the suite's call on a mostly accepted stream) the confusion matrices come from the
//     boundary rows afterwards (confusion_from_rows_kernel, confusion_fix_kernel for the items the certificate rejects).
//   * per item and warp: column totals -> |thickness diff|, boundary error sums (REDUX warp sums), private
//     histograms -> K x K counts; the strips of an item meet in the zero-initialised outputs through
//     global reductions (a few dozen RED per warp and item), never at a CTA barrier.
//
// WIDE KERNEL (K <= 16, W % 4 == 0): warp per 128-column strip, run-length scan with per-lane run queues drained in
// lockstep (label_pass_wide below).
// GENERIC KERNEL: any H, W, K <= 16: thread per column, run-length accumulation down the column.
#include <cuda.h>      // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)

#include <cstdlib>

#include "common.cuh"

namespace octm {

constexpr int kStrip = 128;        // columns per consumer warp
constexpr int kQueueCap = 64;      // queue entries (16 pixel pairs each) per warp
constexpr uint32_t kPadWord = 0x08080808u;   // label 8: PRMT nibble 8 = "replicate sign of LUT byte 0" = 0x00
constexpr uint32_t kSkipWord = 0xFFFFFFFFu;  // queue marker: this word holds no pixels
// unsorted[item] bit 2, set by the label pass without the histogram when the item has a label >= K and cleared by
// confusion_fix_kernel, which counts such items pixel by pixel; callers only ever see bits 0 and 1
constexpr uint32_t kBadLabels = 4u;

struct LabelPassParams {
    const uint8_t* yt;
    const uint8_t* yp;
    long long n_items;
    int H, W, K;
    int R;   // rows per stage, multiple of 4
    int S;   // ring stages
    unsigned long long* counts;
    long long* thick;
    long long* bsq;
    long long* babs;
    int* bnd_t;
    int* bnd_p;
    unsigned* first_pos;
    unsigned* unsorted;   // [n] bit 0 / 1: some column of y_true / y_pred is not non-decreasing from top to bottom (or null)
    uint32_t one;   // always 1, but opaque to ptxas: `x * one + y` is then an IMAD on the (idle) FMA pipe
                    // instead of an IADD3 on the ALU pipe that the PRMT-heavy inner loop saturates
};

// shared-memory carve-up of the fast kernel

constexpr int kOffWarp = 0;          // no CTA-wide block any more: warps are autonomous
constexpr int kWarpTotals = 2 * 8 * kStrip * 2;    // u16 [map][thr][128]
constexpr int kWarpHist = 64 * 32 * 2;             // u16 [code][lane]
constexpr int kWarpQueue = kQueueCap * 16;         // uint4 entries
constexpr int kWarpBars = 768;                     // the warp's S "stage full" mbarriers (64 B), flags (at +64), first-position
                                                   // table (128 B at +128), last rows of the lanes' mixed passes (512 B at +256)
constexpr int kWarpBytesShort = kWarpHist + kWarpQueue;              // H <= 500: totals alias the histogram block
constexpr int kWarpBytesTall = kWarpHist + kWarpQueue + kWarpTotals;
// The byte counters are flushed after every 18 x 7 four-row groups, the last of which may be partial: an item of more
// than 500 rows (126 groups) is flushed before its epilogue, and the flush would land in the histogram block the
// totals of shorter items alias (and leave nothing for the certificate's byte-counter check).
constexpr int kShortRows = 500;

// PRMT look-up words for threshold pair q (k1 = 2q+1, k2 = 2q+2); byte i describes label v0 + i.
//   q <  2 : flags [v <  k1] | [v <  k2] << 4  -- non-zero only for labels 0-3
//   q >= 2 : flags [v >= k1] | [v >= k2] << 4  -- non-zero only for labels 4-7
// The SASS PRMT takes an immediate only as its second data word (labels 4-7), and ptxas re-materialises a
// register constant before every use, so the "below" pairs are looked up with the selector + 4 per
// nibble: labels 0-3 then pick the immediate word, labels 4-7 (nibble 8-11) and the pad label (nibble 12)
// pick a replicated sign bit of a zero byte.  No look-up constant lives in a register.
// The epilogue turns the "below" counts of thresholds 1-4 back into "at or above" (H - count).
__host__ __device__ constexpr uint32_t lut_word(int q, int v0) {
    const int k1 = 2 * q + 1, k2 = 2 * q + 2;
    uint32_t w = 0;
    for (int i = 0; i < 4; ++i) {
        int v = v0 + i;
        uint32_t b = q < 2 ? ((v < k1 ? 1u : 0u) | (v < k2 ? 0x10u : 0u)) : ((v >= k1 ? 1u : 0u) | (v >= k2 ? 0x10u : 0u));
        w |= b << (8 * i);
    }
    return w;
}
constexpr int kBelowThresholds = 4;   // thresholds 1..4 are counted as "label below"

// raw PRMT: unlike __byte_perm the selector is not masked to 3 bits per nibble, so nibble value 8
// (the pad label) selects "sign of byte 0", which is 0x00 for every LUT used here.
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

__device__ __forceinline__ uint2 lds64(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}

// Column-scan state of one lane: 2 word slots x 2 halves; every accumulator byte belongs to one
// (map, column): byte0 = y_true col a, byte1 = y_pred col a, byte2 = y_true col b, byte3 = y_pred col b,
// with (a, b) = columns (0, 1) of the word for half 0 and (2, 3) for half 1.
template <int NP>
struct ColState {
    uint32_t nib[2][2][NP];        // two 4-bit counters per byte: thresholds 2q+1 (low), 2q+2 (high)
    uint32_t byt[2][2][2 * NP];    // one 8-bit counter per byte: threshold j+1
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int s = 0; s < 2; ++s)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
#pragma unroll
                for (int q = 0; q < NP; ++q) nib[s][h][q] = 0;
#pragma unroll
                for (int j = 0; j < 2 * NP; ++j) byt[s][h][j] = 0;
            }
    }
    __device__ __forceinline__ void nib_to_byte() {
#pragma unroll
        for (int s = 0; s < 2; ++s)
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int q = 0; q < NP; ++q) {
                    byt[s][h][2 * q] += nib[s][h][q] & 0x0f0f0f0fu;
                    byt[s][h][2 * q + 1] += (nib[s][h][q] >> 4) & 0x0f0f0f0fu;
                    nib[s][h][q] = 0;
                }
    }
    // add the byte counters into the warp's uint16 column totals [map][thr][128] and clear them
    __device__ __forceinline__ void byte_to_totals(unsigned short* totals, int lane) {
#pragma unroll
        for (int hp = 0; hp < 2; ++hp) {          // the two row phases own the same columns: take turns
            if ((lane >> 4) == hp) {
#pragma unroll
                for (int j = 0; j < 2 * NP; ++j) {
                    uint4* tt = reinterpret_cast<uint4*>(totals + (0 * 8 + j) * kStrip + (lane & 15) * 8);
                    uint4* tp = reinterpret_cast<uint4*>(totals + (1 * 8 + j) * kStrip + (lane & 15) * 8);
                    uint4 a = *tt, b = *tp;
                    a.x += prmt(byt[0][0][j], 0, 0x4240); b.x += prmt(byt[0][0][j], 0, 0x4341);
                    a.y += prmt(byt[0][1][j], 0, 0x4240); b.y += prmt(byt[0][1][j], 0, 0x4341);
                    a.z += prmt(byt[1][0][j], 0, 0x4240); b.z += prmt(byt[1][0][j], 0, 0x4341);
                    a.w += prmt(byt[1][1][j], 0, 0x4240); b.w += prmt(byt[1][1][j], 0, 0x4341);
                    *tt = a;
                    *tp = b;
                    byt[0][0][j] = byt[0][1][j] = byt[1][0][j] = byt[1][1][j] = 0;
                }
            }
            __syncwarp();
        }
    }
};

// two rows (A, B) of one word slot: t/p words -> interleaved selector -> LUT flags -> nibble counters
template <int NP>
__device__ __forceinline__ void col_accumulate(uint32_t (&nib)[2][NP], uint32_t tA, uint32_t pA, uint32_t tB,
                                               uint32_t pB, uint32_t one) {
    const uint32_t xa = pA * 16u + tA, xb = pB * 16u + tB;      // nibbles: t0 p0 t1 p1 | t2 p2 t3 p3
    const uint32_t sel[2][2] = {{xa, xa >> 16}, {xb, xb >> 16}};
    const uint32_t sel4[2][2] = {{xa * one + 0x44444444u, sel[0][1] * one + 0x4444u},
                                 {xb * one + 0x44444444u, sel[1][1] * one + 0x4444u}};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int q = 0; q < NP; ++q) {
            const uint32_t fa = q < 2 ? prmt(0u, lut_word(q, 0), sel4[0][h]) : prmt(0u, lut_word(q, 4), sel[0][h]);
            const uint32_t fb = q < 2 ? prmt(0u, lut_word(q, 0), sel4[1][h]) : prmt(0u, lut_word(q, 4), sel[1][h]);
            nib[h][q] = fb * one + (fa * one + nib[h][q]);
        }
    }
}

// classes present among one lane's 16 pixel pairs: bits 0-7 y_true, bits 8-15 y_pred (pad label 8 -> none)
__device__ __forceinline__ uint32_t presence_bits(uint2 tA, uint2 pA, uint2 tB, uint2 pB) {
    const uint32_t x0 = pA.x * 16u + tA.x, x1 = pA.y * 16u + tA.y, x2 = pB.x * 16u + tB.x, x3 = pB.y * 16u + tB.y;
    const uint32_t lo = 0x08040201u, hi = 0x80402010u;
    const uint32_t w = (prmt(lo, hi, x0) | prmt(lo, hi, x0 >> 16)) | (prmt(lo, hi, x1) | prmt(lo, hi, x1 >> 16)) |
                       (prmt(lo, hi, x2) | prmt(lo, hi, x2 >> 16)) | (prmt(lo, hi, x3) | prmt(lo, hi, x3 >> 16));
    return (w | (w >> 16)) & 0xffffu;
}

// index (0-7) of the first byte equal to c in the 8 labels {w.x, w.y}, or 8
__device__ __forceinline__ uint32_t first_match8(uint2 w, uint32_t cc) {
    const uint32_t z0 = ~((w.x ^ cc) + 0x7f7f7f7fu) & 0x80808080u;   // labels < 16: exact zero-byte test
    const uint32_t z1 = ~((w.y ^ cc) + 0x7f7f7f7fu) & 0x80808080u;
    if (z0) return (__ffs(z0) - 1) >> 3;
    if (z1) return 4 + ((__ffs(z1) - 1) >> 3);
    return 8;
}

// a lane met classes `fresh` (bits as presence_bits) for the first time in this item: fold the raster
// position of their first pixel among its rows A (at posA) and B (at posB) into the CTA's table
__device__ __forceinline__ void record_first(uint32_t fresh, uint2 tA, uint2 pA, uint2 tB, uint2 pB, uint32_t posA,
                                             uint32_t posB, uint32_t* first_tab) {
    while (fresh) {
        const int bit = __ffs(fresh) - 1;
        fresh &= fresh - 1;
        const int m = bit >> 3, c = bit & 7;
        const uint32_t cc = 0x01010101u * c;
        uint32_t i = first_match8(m ? pA : tA, cc), pos = posA + i;
        if (i == 8) {
            i = first_match8(m ? pB : tB, cc);
            pos = posB + i;
        }
        if (i < 8 && pos < first_tab[m * 16 + c]) atomicMin(&first_tab[m * 16 + c], pos);
    }
}

// some label among the 8 of one row of both maps (words t, p) is >= K; k_add = (128 - K) per byte
template <int NP>
__device__ __forceinline__ bool labels_from_k(uint2 t, uint2 p, uint32_t k_add) {
    if (NP == 4) return ((t.x | t.y) | (p.x | p.y)) & 0xf8f8f8f8u;      // K = 8: a bit above the 3-bit class range
    // bit 7 of a byte: the label is >= 128, or its low 7 bits plus 128 - K reach 128 (no carry leaves the byte)
    const uint32_t m = (((t.x & 0x7f7f7f7fu) + k_add) | t.x) | (((t.y & 0x7f7f7f7fu) + k_add) | t.y) |
                       (((p.x & 0x7f7f7f7fu) + k_add) | p.x) | (((p.y & 0x7f7f7f7fu) + k_add) | p.y);
    return m & 0x80808080u;
}

__device__ __forceinline__ void hist_add(unsigned short* hist_lane, uint32_t code, uint32_t inc) {
    unsigned short* h = hist_lane + code * 32;
    *h = static_cast<unsigned short>(*h + inc);
}

__device__ __forceinline__ void drain_entry(unsigned short* hist_lane, uint4 e) {
    const uint32_t w[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (w[k] != kSkipWord) {
#pragma unroll
            for (int i = 0; i < 4; ++i) hist_add(hist_lane, (w[k] >> (8 * i)) & 0x3fu, 1);
        }
    }
}

// confusion machinery for up to two rows (16 pixel pairs) of one lane.  j* are joint-code words
// (t*8+p per byte) or kSkipWord for rows that do not exist.
__device__ __forceinline__ void conf_push(bool mixed_lane, uint4 e, unsigned short* hist_lane, uint4* queue,
                                          uint32_t& qhead, uint32_t& qtail, int lane) {
    const uint32_t mixed = __ballot_sync(0xffffffffu, mixed_lane);
    if (mixed) {
        if (mixed_lane) queue[(qtail + __popc(mixed & lanemask_lt())) & (kQueueCap - 1)] = e;
        qtail += __popc(mixed);
        __syncwarp();
        if (qtail - qhead >= 32) {
            drain_entry(hist_lane, queue[(qhead + lane) & (kQueueCap - 1)]);
            qhead += 32;
            __syncwarp();
        }
    }
}

// per-lane running state of one item
template <int NP>
struct LaneState {
    ColState<NP> cs;
    uint32_t qhead, qtail;
    uint32_t last_b;      // joint code (byte-replicated) of this lane's current run of uniform row pairs
    uint32_t run;         // pixel pairs of that run not yet in the histogram
    uint32_t warp_seen;   // classes this warp has met in this item (presence_bits layout, warp-uniform)
    int nib_fill, byt_fill;
    __device__ __forceinline__ void reset(bool cols) {
        if (cols) cs.clear();
        qhead = qtail = 0;
        last_b = 0xffffffffu;
        run = 0;
        warp_seen = 0;
        nib_fill = byt_fill = 0;
    }
};

struct StageConsts {
    uint32_t srow2, srow4;        // 2 / 4 rows of a staged strip in shared memory (bytes)
    uint32_t W2, W4;              // 2 / 4 rows of the image (raster positions)
    uint32_t map_bytes, one, all_classes, k_add;
    int phase, lane;
    bool colv;
    unsigned short* hist_lane;
    uint4* queue;
    unsigned short* totals;
    uint32_t* first_tab;
    uint32_t* bad;                // set when a label with bits above the 3-bit class range shows up
    uint32_t* unsorted;           // bit 0 / 1: a column of y_true / y_pred decreases somewhere (this warp, this item)
    uint4* prev_rows;             // [32] last row (t.x, t.y, p.x, p.y) of a lane's latest mixed pass
};

// One ring stage (rows x strip) of one consumer warp.  Each pass of the loop takes 4 rows: lanes 0-15 rows
// (4i, 4i+2), lanes 16-31 rows (4i+1, 4i+3), 8 columns per lane, both maps.  FULL: every lane has both rows
// (no predicates); otherwise missing rows / columns are replaced by the pad label.
// Kept rolled: one pass is ~100 instructions and must stay inside the L0 instruction cache.
template <int NP, bool CONF, bool COLS, bool SEEDS, bool SORT, bool FULL>
__device__ __forceinline__ void stage_rows(LaneState<NP>& ls, uint32_t at, uint32_t pos, int rows, const StageConsts& sc) {
    const int npairs = (rows + 3) >> 2;
#pragma unroll 1
    for (int pr = 0; pr < npairs; ++pr, at += sc.srow4, pos += sc.W4) {
        uint2 tA, pA, tB, pB;
        bool va = true, vb = true;
        if (FULL) {
            tA = lds64(at);
            tB = lds64(at + sc.srow2);
            pA = lds64(at + sc.map_bytes);
            pB = lds64(at + sc.map_bytes + sc.srow2);
        } else {
            va = sc.colv && 4 * pr + sc.phase < rows;
            vb = sc.colv && 4 * pr + sc.phase + 2 < rows;
            tA = make_uint2(kPadWord, kPadWord); pA = tA; tB = tA; pB = tA;
            if (va) { tA = lds64(at); pA = lds64(at + sc.map_bytes); }
            if (vb) { tB = lds64(at + sc.srow2); pB = lds64(at + sc.map_bytes + sc.srow2); }
        }
        if (COLS) {
            col_accumulate<NP>(ls.cs.nib[0], tA.x, pA.x, tB.x, pB.x, sc.one);
            col_accumulate<NP>(ls.cs.nib[1], tA.y, pA.y, tB.y, pB.y, sc.one);
        }
        if (CONF || SEEDS || SORT) {
            uint4 j = make_uint4(tA.x * 8u + pA.x, tA.y * 8u + pA.y, tB.x * 8u + pB.x, tB.y * 8u + pB.y);
            const uint32_t b = prmt(j.x, 0, 0);
            // labels >= 8 (outside what the 6-bit joint code can hold) must never alias a valid code: OR of all 16
            // label pairs, bits 3-7 of every byte (the pad label 8 of missing rows / columns is masked out below)
            const uint32_t high = ((tA.x | tA.y | tB.x) | (tB.y | pA.x | pA.y) | (pB.x | pB.y)) & 0xf8f8f8f8u;
            // uniform lane: all 16 pixel pairs share one joint code (padded lanes never take this path)
            const bool uni = FULL && ((((j.x ^ b) | (j.y ^ b)) | ((j.z ^ b) | (j.w ^ b))) | high) == 0;
            // uniform row pairs come in long runs of one joint code (a lane stays inside a layer for many rows): the
            // run length lives in a register and reaches the lane's private histogram column when the code changes
            const bool changed = uni && b != ls.last_b;
            if (CONF && uni && !changed) ls.run += 16u;
            const bool mixed_lane = FULL ? !uni : (va || vb);
            if (__any_sync(0xffffffffu, mixed_lane || changed)) {
                if (SORT && (mixed_lane || changed)) {
                    // Column order, part 1 of 2: along THIS lane's own rows (every other row of its 8 columns) the
                    // labels must not decrease: previous row <= A <= B, bytewise, both maps.  Uniform unchanged
                    // passes need no check (same labels as the row before); the row before a checked pass is the
                    // open run's code, or -- after a mixed pass, which closes the run -- the copy in shared memory.
                    // Part 2 (the two row parities interleave) is the count comparison in the item epilogue.
                    uint32_t t0, t1, p0, p1;
                    if (ls.last_b == 0xffffffffu) {
                        const uint4 v = sc.prev_rows[sc.lane];
                        t0 = v.x; t1 = v.y; p0 = v.z; p1 = v.w;
                    } else {
                        t0 = t1 = (ls.last_b >> 3) & 0x07070707u;
                        p0 = p1 = ls.last_b & 0x07070707u;
                    }
                    const uint32_t M = 0x80808080u;       // (a | M) - b keeps bit 7 of a byte iff a >= b (labels < 128)
                    const uint32_t gt = ((tA.x | M) - t0) & ((tA.y | M) - t1) & ((tB.x | M) - tA.x) & ((tB.y | M) - tA.y) & M;
                    const uint32_t gp = ((pA.x | M) - p0) & ((pA.y | M) - p1) & ((pB.x | M) - pA.x) & ((pB.y | M) - pA.y) & M;
                    if (gt != M || gp != M) atomicOr(sc.unsorted, (gt != M ? 1u : 0u) | (gp != M ? 2u : 0u));
                    if (mixed_lane) {                     // close the run: the next pass of this lane is checked against B
                        if (CONF && ls.last_b != 0xffffffffu) hist_add(sc.hist_lane, ls.last_b & 0x3fu, ls.run);
                        ls.last_b = 0xffffffffu;
                        ls.run = 0;
                        sc.prev_rows[sc.lane] = make_uint4(tB.x, tB.y, pB.x, pB.y);
                    }
                }
                if (CONF && (FULL ? high != 0 : ((va && ((tA.x | tA.y | pA.x | pA.y) & 0xf8f8f8f8u)) ||
                                        (vb && ((tB.x | tB.y | pB.x | pB.y) & 0xf8f8f8f8u)))))
                    *sc.bad = 1;                    // this warp's counts of the item are withheld (epilogue)
                // without the histogram the item's counts come from its boundary rows, which cannot see a label >= K:
                // such an item is sent to the per-pixel histogram instead (a uniform lane's labels are checked when
                // its run starts, so checking the lanes of this block covers every pixel)
                if (!CONF && SORT && ((va && labels_from_k<NP>(tA, pA, sc.k_add)) || (vb && labels_from_k<NP>(tB, pB, sc.k_add))))
                    atomicOr(sc.unsorted, kBadLabels);
                if (changed) {
                    if (CONF && ls.last_b != 0xffffffffu) hist_add(sc.hist_lane, ls.last_b & 0x3fu, ls.run);
                    ls.last_b = b;
                    ls.run = 16u;
                }
                if (SEEDS) {
                    // classes are tracked per WARP: rows only grow from pass to pass, so once any lane has
                    // met a class, later passes cannot hold an earlier pixel of it
                    uint32_t fresh = 0;
                    if ((changed || mixed_lane) && ls.warp_seen != sc.all_classes) {
                        const uint32_t bits = uni ? ((1u << ((b >> 3) & 7u)) | (0x100u << (b & 7u)))
                                                  : presence_bits(tA, pA, tB, pB);
                        fresh = bits & ~ls.warp_seen;
                    }
                    const uint32_t any_fresh = __reduce_or_sync(0xffffffffu, fresh);
                    if (any_fresh) {
                        ls.warp_seen |= any_fresh;
                        if (fresh) record_first(fresh, tA, pA, tB, pB, pos, pos + sc.W2, sc.first_tab);
                    }
                }
                __syncwarp();
                if (CONF) {
                    if (!FULL) {
                        if (!va) j.x = j.y = kSkipWord;
                        if (!vb) j.z = j.w = kSkipWord;
                    }
                    conf_push(mixed_lane, j, sc.hist_lane, sc.queue, ls.qhead, ls.qtail, sc.lane);
                }
            }
        }
        if (COLS && ++ls.nib_fill == 7) {
            ls.cs.nib_to_byte();
            ls.nib_fill = 0;
            if (++ls.byt_fill == 18) { ls.byt_fill = 0; ls.cs.byte_to_totals(sc.totals, sc.lane); }
        }
    }
}

// Shared memory of the fast kernel: a fixed CTA block (kOffWarp bytes), then one private block per warp:
//   [ S full-barriers, padded to 128 B | histogram 4 KB | queue 1 KB | (H > 500: column totals 4 KB) | ring ]
// The ring is PRIVATE to the warp: S stages x 2 maps x R rows x strip bytes, filled by 2-D TMA tile copies
// (one box of R rows x 128 columns per map) that the warp issues for itself.  Warps of a CTA therefore
// never wait for each other: each folds its strip's results into the zero-initialised outputs with global
// reductions (RED.ADD / RED.MIN), so a CTA has no barrier after its start-up.
template <int NP, bool CONF, bool COLS, bool SEEDS, bool SORT, bool WIDE>
__global__ void __launch_bounds__(WIDE ? 16 * 32 : 8 * 32, WIDE ? 1 : 2)
label_pass_fast(const LabelPassParams prm, const __grid_constant__ CUtensorMap tm_true, const __grid_constant__ CUtensorMap tm_pred) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NW = blockDim.x >> 5;
    const int H = prm.H, W = prm.W, K = prm.K, R = prm.R, S = prm.S;

    const bool tall = H > kShortRows;
    const uint32_t srow = static_cast<uint32_t>(min(W, kStrip));          // bytes per staged strip row
    const uint32_t map_bytes = static_cast<uint32_t>(R) * srow;
    const uint32_t stage_bytes = 2 * map_bytes;
    const int state_bytes = kWarpBars + (tall ? kWarpBytesTall : kWarpBytesShort);
    const int warp_bytes = state_bytes + S * static_cast<int>(stage_bytes);   // multiple of 128

    uint8_t* wbase = smem + kOffWarp + warp * warp_bytes;
    for (int i = lane; i < state_bytes / 4; i += 32) reinterpret_cast<uint32_t*>(wbase)[i] = 0;
    const uint32_t bars = smem_u32(wbase);                                  // full[s] at bars + 8 s
    const uint32_t ring_addr = bars + state_bytes;
    uint32_t* warp_first = reinterpret_cast<uint32_t*>(wbase + 128);        // [2][16] first raster position per class
    uint32_t* warp_bad = reinterpret_cast<uint32_t*>(wbase + 64);           // a label >= 8 was met in this item
    uint32_t* warp_unsorted = reinterpret_cast<uint32_t*>(wbase + 68);      // bit 0 / 1: a column of y_true / y_pred is out of order
    uint4* prev_rows = reinterpret_cast<uint4*>(wbase + 256);               // [32]
    if (lane == 0) {
        for (int s = 0; s < S; ++s) mbar_init_a(bars + 8 * s, 1);
        mbar_fence_init();
    }
    __syncthreads();

    // ---------------------------------------------------------------------- ring fills (per warp)
    // The warp's stages form one fixed sequence (item by item, R rows at a time); fill f lives in slot
    // f % S and is issued by lane 0 right after fill f - S has been consumed.  A box always has R rows:
    // past the end of an item it carries rows of the next one (never read), past the end of the tensor zeros.
    const uint64_t pol = policy_evict_first();
    const int x0 = warp * kStrip;
    auto issue_fill = [&](long long it, int r0, uint32_t slot) {
        const uint32_t dst = ring_addr + slot * stage_bytes;
        const int y = static_cast<int>(it * H + r0);
        mbar_expect_tx_a(bars + 8 * slot, stage_bytes);
        tma_load_2d(dst, &tm_true, x0, y, bars + 8 * slot, pol);
        tma_load_2d(dst + map_bytes, &tm_pred, x0, y, bars + 8 * slot, pol);
    };
    long long nf_item = blockIdx.x;
    int nf_r0 = 0;
    for (int f = 0; f < S; ++f) {
        if (lane == 0 && nf_item < prm.n_items) issue_fill(nf_item, nf_r0, f);
        nf_r0 += R;
        if (nf_r0 >= H) { nf_r0 = 0; nf_item += gridDim.x; }
    }

    // ---------------------------------------------------------------------- consumers
    unsigned short* hist = reinterpret_cast<unsigned short*>(wbase + kWarpBars);             // [64][32]
    unsigned short* hist_lane = hist + lane;
    uint4* queue = reinterpret_cast<uint4*>(wbase + kWarpBars + kWarpHist);
    unsigned short* totals = tall ? reinterpret_cast<unsigned short*>(wbase + kWarpBars + kWarpHist + kWarpQueue) : hist;   // [2][8][128]
    const int phase = lane >> 4;
    const int col = warp * kStrip + (lane & 15) * 8;      // first of this lane's 8 columns
    const bool colv = col < W;
    const bool strip_full = (warp + 1) * kStrip <= W;      // warp-uniform
    const int nthr = K - 1;
    const uint32_t lane_smem = static_cast<uint32_t>(phase) * srow + (lane & 15) * 8;     // inside a staged strip
    const uint32_t lane_pos = static_cast<uint32_t>(phase) * W + col;                       // inside the image

    StageConsts sc;
    sc.srow2 = 2u * srow; sc.srow4 = 4u * srow; sc.W2 = 2u * W; sc.W4 = 4u * W;
    sc.map_bytes = map_bytes; sc.one = prm.one; sc.all_classes = ((1u << K) - 1u) * 0x101u;
    sc.k_add = static_cast<uint32_t>(128 - K) * 0x01010101u;
    sc.phase = phase; sc.lane = lane; sc.colv = colv;
    sc.hist_lane = hist_lane; sc.queue = queue; sc.totals = totals; sc.first_tab = warp_first; sc.bad = warp_bad;
    sc.unsorted = warp_unsorted; sc.prev_rows = prev_rows;
    LaneState<NP> ls;
    uint32_t s = 0, ph = 0;
    for (long long item = blockIdx.x; item < prm.n_items; item += gridDim.x) {
        ls.reset(COLS);
        if (CONF && lane == 0) *warp_bad = 0;
        if (SORT) {
            if (lane == 0) *warp_unsorted = tall ? 3u : 0u;      // items that flush their byte counters: not certified
            prev_rows[lane] = make_uint4(0, 0, 0, 0);
        }
        if (SEEDS) warp_first[lane] = OCTM_NO_SEED;
        __syncwarp();

        for (int r0 = 0; r0 < H; r0 += R) {
            const int rows = min(R, H - r0);
            mbar_wait_parked_a(bars + 8 * s, ph);
            const uint32_t at = ring_addr + s * stage_bytes + lane_smem;        // this lane's first row, y_true
            const uint32_t pos = static_cast<uint32_t>(r0) * W + lane_pos;       // its raster index in the item
            if (strip_full && (rows & 3) == 0)       // warp-uniform: every lane has both of its rows
                stage_rows<NP, CONF, COLS, SEEDS, SORT, true>(ls, at, pos, rows, sc);
            else                                     // ragged strip or last rows of the item
                stage_rows<NP, CONF, COLS, SEEDS, SORT, false>(ls, at, pos, rows, sc);
            __syncwarp();                            // every lane has read the slot
            if (lane == 0 && nf_item < prm.n_items) {
                fence_proxy_async();                 // generic reads of the slot before the async overwrite
                issue_fill(nf_item, nf_r0, s);
            }
            nf_r0 += R;
            if (nf_r0 >= H) { nf_r0 = 0; nf_item += gridDim.x; }
            if (++s == static_cast<uint32_t>(S)) { s = 0; ph ^= 1; }
        }

        // ------------------------------------------------------------------ item epilogue
        // The histogram fold runs first and leaves its shared-memory block zeroed: for items of at most
        // kShortRows rows (no byte flush before the epilogue) the column totals reuse that block.
        if (CONF) {
            // leftover queue entries, then fold the 32 private histogram columns
            if (ls.last_b != 0xffffffffu) hist_add(hist_lane, ls.last_b & 0x3fu, ls.run);      // the open run
            const uint32_t left = ls.qtail - ls.qhead;
            __syncwarp();
            if (static_cast<uint32_t>(lane) < left) drain_entry(hist_lane, queue[(ls.qhead + lane) & (kQueueCap - 1)]);
            __syncwarp();
            // a label >= 8 may have aliased a valid joint code: withhold this warp's counts, so that the item's
            // confusion matrix does not add up to H * W and the epilogue reports it (labels in [K, 8) are dropped
            // by the t < K && pp < K test below: same effect)
            const bool wbad = *warp_bad != 0;
            uint32_t* h32 = reinterpret_cast<uint32_t*>(hist);
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                const int code = lane * 2 + cc;
                uint32_t lo = 0, hi = 0;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int j = (lane + i) & 15;
                    const uint32_t w = h32[code * 16 + j];
                    h32[code * 16 + j] = 0;
                    lo += w & 0xffffu;
                    hi += w >> 16;
                }
                // this warp's share of cm[t][p] joins the other strips' in the (zero-initialised) output
                const int t = code >> 3, pp = code & 7;
                if ((lo + hi) && t < K && pp < K && !wbad && prm.counts != nullptr)
                    atomicAdd(prm.counts + (item * K + t) * K + pp, static_cast<unsigned long long>(lo + hi));
            }
        }

        __syncwarp();
        if (COLS) {
            ls.cs.nib_to_byte();
            if (SORT && !tall) {
                // Column order, part 2 of 2.  Lanes l and l ^ 16 hold the counts of the even and of the odd rows of
                // the same 8 columns.  Each parity's rows are in order (part 1), so the whole column is in order iff
                // for every threshold k  #{even rows below k} - #{odd rows below k} is 0 or 1  (the rows below k
                // then form a prefix of the column).  Thresholds counted as "at or above" mirror this.
                uint32_t viol_t = 0, viol_p = 0;
                const bool h_even = (H & 1) == 0;
#pragma unroll
                for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                        for (int j = 0; j < 2 * NP; ++j) {
                            const uint32_t mine = ls.cs.byt[sl][hh][j];
                            const uint32_t other = __shfl_xor_sync(0xffffffffu, mine, 16);      // odd rows, seen from phase 0
                            const bool below = j < kBelowThresholds;
                            const uint32_t a = (below || !h_even) ? mine : other, b = (below || !h_even) ? other : mine;
                            // a - b per byte must be 0 or 1; the two maps' bytes (even: y_true, odd: y_pred) are
                            // subtracted in separate 16-bit fields with a guard bit, so that a borrow stays in its field
                            const uint32_t G = 0x01000100u;
                            const uint32_t dt = ((a & 0x00ff00ffu) | G) - (b & 0x00ff00ffu);
                            const uint32_t dp = (((a >> 8) & 0x00ff00ffu) | G) - ((b >> 8) & 0x00ff00ffu);
                            viol_t |= (dt ^ G) & 0xfffefffeu;
                            viol_p |= (dp ^ G) & 0xfffefffeu;
                        }
                if (phase == 0 && (viol_t | viol_p)) atomicOr(warp_unsorted, (viol_t ? 1u : 0u) | (viol_p ? 2u : 0u));
            }
            ls.cs.byte_to_totals(totals, lane);
            // per-column arithmetic: lane owns 4 columns of the strip
            const int lc = lane * 4;
            const bool cv = warp * kStrip + lc < W;
            uint32_t sq[2 * NP], ab[2 * NP], th[2 * NP + 1];
            uint32_t fkt[2 * NP + 1], fkp[2 * NP + 1];
#pragma unroll
            for (int j = 0; j < 2 * NP + 1; ++j) fkt[j] = fkp[j] = OCTM_NO_SEED;
#pragma unroll
            for (int j = 0; j < 2 * NP; ++j) sq[j] = ab[j] = 0;
#pragma unroll
            for (int j = 0; j < 2 * NP + 1; ++j) th[j] = 0;
            if (cv) {
                // stream over thresholds k = j + 1: cur = #{label >= k} per column, prev = #{label >= k - 1}
                int pvt[4] = {H, H, H, H}, pvp[4] = {H, H, H, H};
                const long long ob = (item * nthr) * W + warp * kStrip + lc;
#pragma unroll
                for (int j = 0; j < 2 * NP; ++j) {
                    uint2* pt = reinterpret_cast<uint2*>(totals + (0 * 8 + j) * kStrip + lc);
                    uint2* pp = reinterpret_cast<uint2*>(totals + (1 * 8 + j) * kStrip + lc);
                    const uint2 a = *pt, b = *pp;
                    *pt = make_uint2(0, 0);
                    *pp = make_uint2(0, 0);
                    int cut[4] = {int(a.x & 0xffff), int(a.x >> 16), int(a.y & 0xffff), int(a.y >> 16)};
                    int cup[4] = {int(b.x & 0xffff), int(b.x >> 16), int(b.y & 0xffff), int(b.y >> 16)};
                    if (j < kBelowThresholds) {      // thresholds 1-4 were counted as "label below"
#pragma unroll
                        for (int i = 0; i < 4; ++i) { cut[i] = H - cut[i]; cup[i] = H - cup[i]; }
                    }
                    if (SORT && !SEEDS) {
                        // first raster position of class j in these columns IF the column is in class order: its pixels
                        // start at row #{label < j} = H - #{label >= j}
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            if (pvt[i] > cut[i]) fkt[j] = min(fkt[j], static_cast<uint32_t>((H - pvt[i]) * W + warp * kStrip + lc + i));
                            if (pvp[i] > cup[i]) fkp[j] = min(fkp[j], static_cast<uint32_t>((H - pvp[i]) * W + warp * kStrip + lc + i));
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int d = cut[i] - cup[i];
                        sq[j] += d * d;
                        ab[j] += abs(d);
                        th[j] += abs((pvt[i] - cut[i]) - (pvp[i] - cup[i]));
                        pvt[i] = cut[i];
                        pvp[i] = cup[i];
                    }
                    if (prm.bnd_t != nullptr && j < nthr) {
                        *reinterpret_cast<int4*>(prm.bnd_t + ob + static_cast<long long>(j) * W) =
                            make_int4(H - cut[0], H - cut[1], H - cut[2], H - cut[3]);
                        *reinterpret_cast<int4*>(prm.bnd_p + ob + static_cast<long long>(j) * W) =
                            make_int4(H - cup[0], H - cup[1], H - cup[2], H - cup[3]);
                    }
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) th[2 * NP] += abs(pvt[i] - pvp[i]);
                if (SORT && !SEEDS) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (pvt[i] > 0) fkt[2 * NP] = min(fkt[2 * NP], static_cast<uint32_t>((H - pvt[i]) * W + warp * kStrip + lc + i));
                        if (pvp[i] > 0) fkp[2 * NP] = min(fkp[2 * NP], static_cast<uint32_t>((H - pvp[i]) * W + warp * kStrip + lc + i));
                    }
                }
            }
            if (SORT && !SEEDS && prm.first_pos != nullptr) {
                // Seeds for free: on a map whose columns are in class order (the certificate) the first pixel of a class is
                // the minimum over the columns of its first row.  Maps that turn out NOT to be in order get their seeds
                // from first_pos_fix_kernel afterwards (a second read of those maps only).
#pragma unroll
                for (int c = 0; c < 2 * NP + 1; ++c) {
                    if (c < K) {
                        const uint32_t a = __reduce_min_sync(0xffffffffu, fkt[c]), b = __reduce_min_sync(0xffffffffu, fkp[c]);
                        if (lane == 0 && a != OCTM_NO_SEED) atomicMin(prm.first_pos + (item * 2 + 0) * K + c, a);
                        if (lane == 0 && b != OCTM_NO_SEED) atomicMin(prm.first_pos + (item * 2 + 1) * K + c, b);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 2 * NP; ++j) {
                if (j < nthr) {
                    const uint32_t s1 = __reduce_add_sync(0xffffffffu, sq[j]);
                    const uint32_t s2 = __reduce_add_sync(0xffffffffu, ab[j]);
                    if (lane == 0) {
                        if (prm.bsq != nullptr && s1) atomicAdd(reinterpret_cast<unsigned long long*>(prm.bsq) + item * nthr + j, static_cast<unsigned long long>(s1));
                        if (prm.babs != nullptr && s2) atomicAdd(reinterpret_cast<unsigned long long*>(prm.babs) + item * nthr + j, static_cast<unsigned long long>(s2));
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < 2 * NP + 1; ++c) {
                if (c < K) {
                    const uint32_t s3 = __reduce_add_sync(0xffffffffu, th[c]);
                    if (lane == 0 && prm.thick != nullptr && s3)
                        atomicAdd(reinterpret_cast<unsigned long long*>(prm.thick) + item * K + c, static_cast<unsigned long long>(s3));
                }
            }
        }
        if (SORT && prm.unsorted != nullptr) {
            __syncwarp();
            if (lane == 0 && *warp_unsorted) atomicOr(prm.unsorted + item, *warp_unsorted);
        }
        if (SEEDS && prm.first_pos != nullptr) {
            __syncwarp();
            const int m = lane >> 4, c = lane & 15;
            const uint32_t v = warp_first[lane];
            if (c < K && v != OCTM_NO_SEED) atomicMin(prm.first_pos + (item * 2 + m) * K + c, v);
        }
    }
}

// ------------------------------------------------------------------------------------ generic
// Any H, W and K <= 16 (the fast kernel takes K <= 8, W % 16 == 0).  One CTA per item (grid-stride); a thread
// walks one column at a time (stride blockDim), so adjacent threads read adjacent bytes of a row.  Down a column
// the joint code (t, p) comes in long RUNS (a column stays inside a layer for many rows): only a run's length
// is accumulated per pixel; when the code changes the run goes into the warp's shared-memory confusion
// histogram (one atomic per run, not per pixel) and into the thread's own per-class column counters.
__global__ void __launch_bounds__(256, 4) label_pass_generic(const LabelPassParams prm, const int strips) {
    __shared__ uint32_t s_counts[8][256];                 // per-warp confusion histogram, code = t * 16 + p
    __shared__ unsigned short s_cls[2][16][256];          // per-thread class counts of the current column
    __shared__ unsigned long long s_sq[16], s_abs[16], s_thick[16];
    __shared__ uint32_t s_first[2][16];
    __shared__ uint32_t s_unsorted;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int H = prm.H, W = prm.W, K = prm.K, nthr = K - 1;
    // strips > 1 (few items): a CTA takes 256 columns of an item and adds its share to zero-initialised outputs
    const long long jobs = prm.n_items * strips;
    for (long long job = blockIdx.x; job < jobs; job += gridDim.x) {
        const long long item = job / strips;
        const int xbeg = strips > 1 ? static_cast<int>(job % strips) * 256 : 0;
        const int xend = strips > 1 ? min(W, xbeg + 256) : W;
        for (int i = tid; i < 8 * 256; i += 256) (&s_counts[0][0])[i] = 0;
        if (tid < 16) s_sq[tid] = s_abs[tid] = s_thick[tid] = 0;
        if (tid < 32) (&s_first[0][0])[tid] = OCTM_NO_SEED;
        if (tid == 0) s_unsorted = 0;
        __syncthreads();
        const uint8_t* bt = prm.yt + item * H * static_cast<long long>(W);
        const uint8_t* bp = prm.yp + item * H * static_cast<long long>(W);
        // a warp takes 32 adjacent columns at a time (uniform trip count: lanes past the last column run on empty counts);
        // their sums meet in a warp reduction and one shared-memory atomic per quantity -- nothing is carried in
        // registers across columns, which is what lets four CTAs share an SM (126 registers, two CTAs before)
        const bool wide = static_cast<unsigned long long>(H) * H * 32ull >= (1ull << 32);
        const int lane = tid & 31;
        for (int x0 = xbeg + warp * 32; x0 < xend; x0 += 256) {
            const int x = x0 + lane;
            const bool valid = x < xend;
#pragma unroll
            for (int c = 0; c < 16; ++c) s_cls[0][c][tid] = s_cls[1][c][tid] = 0;
            if (valid) {
            uint32_t seen_t = 0, seen_p = 0;     // raster index grows with y inside one column
            uint32_t run_code = 0xffffffffu, run = 0;
            auto flush = [&]() {
                // a run with a label >= K is dropped (never aliased into another class): the item's counts then do
                // not add up to H * W, which the epilogue reports
                if (run && (run_code >> 8) < static_cast<uint32_t>(K) && (run_code & 255u) < static_cast<uint32_t>(K)) {
                    const uint32_t t = run_code >> 8, p = run_code & 255u;
                    atomicAdd(&s_counts[warp][t * 16u + p], run);
                    s_cls[0][t][tid] = static_cast<unsigned short>(s_cls[0][t][tid] + run);
                    s_cls[1][p][tid] = static_cast<unsigned short>(s_cls[1][p][tid] + run);
                }
            };
            // the loads of kGenRows rows are issued before any of them is looked at: the run bookkeeping below has
            // shared-memory atomics in it, which the compiler will not move loads across (2 loads in flight per thread
            // otherwise: 280 GB/s)
            constexpr int kGenRows = 8;
            const uint8_t* ct = bt + x;
            const uint8_t* cp = bp + x;
            for (int y0 = 0; y0 < H; y0 += kGenRows) {
                uint32_t tv[kGenRows], pv[kGenRows];
#pragma unroll
                for (int u = 0; u < kGenRows; ++u) {
                    const long long off = static_cast<long long>(min(y0 + u, H - 1)) * W;
                    tv[u] = __ldg(ct + off);
                    pv[u] = __ldg(cp + off);
                }
#pragma unroll
                for (int u = 0; u < kGenRows; ++u) {
                const int y = y0 + u;
                if (y >= H) break;
                const uint32_t t = tv[u], p = pv[u];
                const uint32_t code = t * 256u + p;
                if (code != run_code) {
                    if (run_code != 0xffffffffu && ((t < (run_code >> 8)) || (p < (run_code & 255u))))
                        atomicOr(&s_unsorted, (t < (run_code >> 8) ? 1u : 0u) | (p < (run_code & 255u) ? 2u : 0u));
                    flush();
                    run_code = code;
                    run = 0;
                    if (t < 16u && !((seen_t >> t) & 1u)) {
                        seen_t |= 1u << t;
                        atomicMin(&s_first[0][t], static_cast<uint32_t>(y * W + x));
                    }
                    if (p < 16u && !((seen_p >> p) & 1u)) {
                        seen_p |= 1u << p;
                        atomicMin(&s_first[1][p], static_cast<uint32_t>(y * W + x));
                    }
                }
                ++run;
                }
            }
            flush();
            }
            // column arithmetic from the class counts: #{label >= k} by a suffix sum over the classes
            int ge_t = 0, ge_p = 0;
#pragma unroll 1
            for (int c = K - 1; c >= 0; --c) {
                const int ct = s_cls[0][c][tid], cp = s_cls[1][c][tid];
                const uint32_t th = __reduce_add_sync(0xffffffffu, static_cast<uint32_t>(abs(ct - cp)));
                if (lane == 0 && th) atomicAdd(&s_thick[c], static_cast<unsigned long long>(th));
                ge_t += ct;
                ge_p += cp;
                if (c >= 1) {                                               // threshold k = c
                    const int d = ge_t - ge_p;
                    const uint32_t ab = __reduce_add_sync(0xffffffffu, static_cast<uint32_t>(abs(d)));
                    if (wide) {
                        if (d) atomicAdd(&s_sq[c - 1], static_cast<unsigned long long>(static_cast<long long>(d) * d));
                    } else {
                        const uint32_t sq = __reduce_add_sync(0xffffffffu, static_cast<uint32_t>(d * d));
                        if (lane == 0 && sq) atomicAdd(&s_sq[c - 1], static_cast<unsigned long long>(sq));
                    }
                    if (lane == 0 && ab) atomicAdd(&s_abs[c - 1], static_cast<unsigned long long>(ab));
                    if (valid && prm.bnd_t != nullptr) {
                        prm.bnd_t[(item * nthr + (c - 1)) * W + x] = H - ge_t;
                        prm.bnd_p[(item * nthr + (c - 1)) * W + x] = H - ge_p;
                    }
                }
            }
        }
        __syncthreads();
        if (prm.counts != nullptr) {
            for (int i = tid; i < K * K; i += 256) {
                const int code = (i / K) * 16 + (i % K);
                unsigned long long sum = 0;
                for (int w = 0; w < 8; ++w) sum += s_counts[w][code];
                if (strips == 1) prm.counts[item * K * K + i] = sum;
                else if (sum) atomicAdd(prm.counts + item * K * K + i, sum);
            }
        }
        if (strips == 1) {
            if (tid < K && prm.thick != nullptr) prm.thick[item * K + tid] = static_cast<long long>(s_thick[tid]);
            if (tid < nthr && prm.bsq != nullptr) prm.bsq[item * nthr + tid] = static_cast<long long>(s_sq[tid]);
            if (tid < nthr && prm.babs != nullptr) prm.babs[item * nthr + tid] = static_cast<long long>(s_abs[tid]);
        } else {
            if (tid < K && prm.thick != nullptr && s_thick[tid])
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.thick) + item * K + tid, s_thick[tid]);
            if (tid < nthr && prm.bsq != nullptr && s_sq[tid])
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.bsq) + item * nthr + tid, s_sq[tid]);
            if (tid < nthr && prm.babs != nullptr && s_abs[tid])
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.babs) + item * nthr + tid, s_abs[tid]);
        }
        if (tid == 0 && prm.unsorted != nullptr && s_unsorted) atomicOr(prm.unsorted + item, s_unsorted);
        if (tid < 32 && prm.first_pos != nullptr) {
            const int m = tid >> 4, c = tid & 15;
            if (c < K) {
                if (strips == 1) prm.first_pos[(item * 2 + m) * K + c] = s_first[m][c];
                else if (s_first[m][c] != OCTM_NO_SEED) atomicMin(prm.first_pos + (item * 2 + m) * K + c, s_first[m][c]);
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------ wide columns (K <= 16)
// The shapes of HC-MS / Duke-style label sets (9-10 classes) that the strip kernel (K <= 8) does not take: H <= 16383,
// K <= 16, W % 4 == 0, 4-byte aligned maps.  Same run-length idea as label_pass_generic, restructured so that the per-pixel
// work is a few instructions per 128 pixels and the per-run work runs with all lanes busy:
//   * a WARP owns a job = (item, 128-column strip): a lane reads 4 adjacent columns with one 32-bit load per map and
//     row (a warp row = one 128-byte line per map), 8 rows x 2 maps in flight per lane, issued before any is used;
//   * the (t, p) codes of the 4 columns are formed two at a time by PRMT (t << 8 | p in each half-word) and compared
//     with the open runs' codes as packed words; a run's length is the difference of row numbers: nothing is counted
//     per pixel;
//   * a lane whose column changes class only PUSHES the finished run {length, column, t, p} onto its own queue in
//     shared memory (six predicated instructions); ALL bookkeeping happens when the queues are drained in lockstep --
//     entry i of every lane at once: confusion histogram (one shared atomic per run), the columns' class counts, the
//     order check against the column's previous run and the first positions (private per-lane minima, no atomics;
//     a column's row position is the sum of its runs so far).  Doing the bookkeeping where the change is met costs a
//     divergent pass per row on which ANY of the 128 columns changes -- on tilted layers nearly every row (ncu: 0.67
//     warp-instructions per pixel pair, the same as the byte-wise kernel);
//   * column arithmetic, boundary rows (16-byte stores) and seeds follow per job; warps never meet: their results
//     join in zero-initialised outputs through global atomics (a few hundred per 63 k pixel pairs).
constexpr int kWideWarps = 2;
constexpr int kWideQueue = 48;      // queue entries per lane; a batch of 8 rows pushes at most 32
// per warp: counts u32 [256] | cls u16 [2][K][128] | queue u32 [kWideQueue][32] | fst u32 [2 K][32] | colstate u32 [4][32]
// (sized by K: 17 KB per warp at K = 10 -> 12 warps per SM)
static inline int wide_warp_bytes(int K) { return 1024 + 512 * K + kWideQueue * 128 + 256 * K + 512; }
__global__ void __launch_bounds__(kWideWarps * 32, 7) label_pass_wide(const LabelPassParams prm, const int strips) {
    extern __shared__ __align__(16) unsigned char s_wide[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int H = prm.H, W = prm.W, K = prm.K, nthr = K - 1;
    unsigned char* base = s_wide + warp * (1024 + 512 * K + kWideQueue * 128 + 256 * K + 512);
    uint32_t* counts = reinterpret_cast<uint32_t*>(base);
    unsigned short* cls = reinterpret_cast<unsigned short*>(base + 1024);             // [(map * K + class) * 128 + column]
    uint32_t* queue = reinterpret_cast<uint32_t*>(base + 1024 + 512 * K) + lane;      // entry i at queue[i * 32]: conflict-free
    uint32_t* fst = reinterpret_cast<uint32_t*>(base + 1024 + 512 * K + kWideQueue * 128) + lane;   // [map * K + class][lane]
    uint32_t* colstate = fst + 2 * K * 32;   // [column][lane]: rows so far (16 bits) | last run's t << 16 | its p << 24
    const uint32_t uK = static_cast<uint32_t>(K);
    const long long jobs = prm.n_items * strips;
    // the warps of a CTA take adjacent strips of one item
    for (long long job = static_cast<long long>(blockIdx.x) * kWideWarps + warp; job < jobs;
         job += static_cast<long long>(gridDim.x) * kWideWarps) {
        const long long item = job / strips;
        const int x = static_cast<int>(job % strips) * 128 + 4 * lane;          // this lane's first column
        const bool valid = x < W;                                               // W % 4 == 0: all four or none
        {
            uint4* z = reinterpret_cast<uint4*>(base);                          // counts + cls: 1024 + 512 K bytes
#pragma unroll 1
            for (int i = 0; i < 2 + K; ++i) z[i * 32 + lane] = make_uint4(0, 0, 0, 0);
#pragma unroll 1
            for (int i = 0; i < 2 * K; ++i) fst[i * 32] = OCTM_NO_SEED;
#pragma unroll
            for (int i = 0; i < 4; ++i) colstate[i * 32] = 0xffff0000u;         // no rows yet, no previous run
        }
        __syncwarp();
        uint32_t uns = 0;
        int qn = 0;
        auto drain = [&]() {                     // all lanes, entry i of every queue at once
            const int most = __reduce_max_sync(0xffffffffu, qn);
#pragma unroll 1
            for (int i = 0; i < most; ++i) {
                if (i < qn) {
                    const uint32_t e = queue[i * 32];
                    const uint32_t t = (e >> 8) & 255u, p = e & 255u, J = (e >> 16) & 3u, len = e >> 18;
                    const uint32_t cs = colstate[J * 32];
                    const uint32_t start = cs & 0xffffu, lt = (cs >> 16) & 255u, lp = cs >> 24;
                    colstate[J * 32] = (start + len) | (t << 16) | (p << 24);
                    if (lt != 255u) uns |= (t < lt ? 1u : 0u) | (p < lp ? 2u : 0u);
                    const uint32_t pos = start * static_cast<uint32_t>(W) + static_cast<uint32_t>(x) + J;
                    const uint32_t col = 4u * lane + J;
                    if (t < uK) {
                        fst[t * 32] = min(fst[t * 32], pos);
                        if (p < uK) {                    // a run with a label >= K is dropped, never aliased
                            atomicAdd(&counts[t * 16u + p], len);
                            unsigned short* a = cls + t * 128u + col;
                            unsigned short* b = cls + (uK + p) * 128u + col;
                            *a = static_cast<unsigned short>(*a + len);
                            *b = static_cast<unsigned short>(*b + len);
                        }
                    }
                    if (p < uK) fst[(uK + p) * 32] = min(fst[(uK + p) * 32], pos);
                }
            }
            qn = 0;
        };
        {
            // lanes past the last column scan the last four columns again and push nothing
            const int xc = valid ? x : W - 4;
            const uint8_t* ct = prm.yt + item * H * static_cast<long long>(W) + xc;
            const uint8_t* cp = prm.yp + item * H * static_cast<long long>(W) + xc;
            constexpr int kRows = 8;
            static_assert(4 * kRows <= kWideQueue, "a batch must fit the queue");
            uint32_t ta[kRows], pa[kRows];
            auto fetch = [&](uint32_t (&tv)[kRows], uint32_t (&pv)[kRows], int y0) {
#pragma unroll
                for (int u = 0; u < kRows; ++u) {        // rows past the end repeat the last row: no change, nothing pushed
                    const long long off = static_cast<long long>(min(y0 + u, H - 1)) * W;
                    tv[u] = __ldg(reinterpret_cast<const uint32_t*>(ct + off));
                    pv[u] = __ldg(reinterpret_cast<const uint32_t*>(cp + off));
                }
            };
            fetch(ta, pa, 0);
            // the runs open at row 0
            uint32_t open01 = prmt(pa[0], ta[0], 0x5140u), open23 = prmt(pa[0], ta[0], 0x7362u);
            int st0 = 0, st1 = 0, st2 = 0, st3 = 0;                    // first rows of the open runs
            auto push = [&](uint32_t old, int& st, int y, uint32_t J) {
                queue[qn * 32] = (static_cast<uint32_t>(y - st) << 18) | (J << 16) | old;
                ++qn;
                st = y;
            };
            auto work = [&](const uint32_t (&tv)[kRows], const uint32_t (&pv)[kRows], int y0) {
#pragma unroll
                for (int u = 0; u < kRows; ++u) {
                    const uint32_t c01 = prmt(pv[u], tv[u], 0x5140u), c23 = prmt(pv[u], tv[u], 0x7362u);
                    const uint32_t d01 = c01 ^ open01, d23 = c23 ^ open23;
                    if (valid && (d01 | d23) != 0u) {
                        const int y = y0 + u;
                        if (d01 & 0xffffu) push(open01 & 0xffffu, st0, y, 0u);
                        if (d01 >> 16) push(open01 >> 16, st1, y, 1u);
                        if (d23 & 0xffffu) push(open23 & 0xffffu, st2, y, 2u);
                        if (d23 >> 16) push(open23 >> 16, st3, y, 3u);
                        open01 = c01;
                        open23 = c23;
                    }
                }
            };
            // three register batches: two are in flight while one is worked on
            uint32_t tb[kRows], pb[kRows], tc[kRows], pc[kRows];
            fetch(tb, pb, kRows);
            for (int y0 = 0; y0 < H; y0 += 3 * kRows) {
                fetch(tc, pc, y0 + 2 * kRows);
                work(ta, pa, y0);
                if (__any_sync(0xffffffffu, qn > kWideQueue - 4 * kRows)) drain();
                fetch(ta, pa, y0 + 3 * kRows);
                work(tb, pb, y0 + kRows);
                if (__any_sync(0xffffffffu, qn > kWideQueue - 4 * kRows)) drain();
                fetch(tb, pb, y0 + 4 * kRows);
                work(tc, pc, y0 + 2 * kRows);
                if (__any_sync(0xffffffffu, qn > kWideQueue - 4 * kRows)) drain();
            }
            if (valid) {                                               // the runs still open at the bottom
                push(open01 & 0xffffu, st0, H, 0u);
                push(open01 >> 16, st1, H, 1u);
                push(open23 & 0xffffu, st2, H, 2u);
                push(open23 >> 16, st3, H, 3u);
            }
            drain();
        }
        __syncwarp();
        // column arithmetic from the class counts: #{label >= k} by a suffix sum over the classes, 4 columns per lane
        {
            int get[4] = {0, 0, 0, 0}, gep[4] = {0, 0, 0, 0};
#pragma unroll 1
            for (int c = K - 1; c >= 0; --c) {
                const uint2 a = *reinterpret_cast<const uint2*>(cls + c * 128 + 4 * lane);
                const uint2 b = *reinterpret_cast<const uint2*>(cls + (K + c) * 128 + 4 * lane);
                const int ctv[4] = {static_cast<int>(a.x & 0xffffu), static_cast<int>(a.x >> 16), static_cast<int>(a.y & 0xffffu), static_cast<int>(a.y >> 16)};
                const int cpv[4] = {static_cast<int>(b.x & 0xffffu), static_cast<int>(b.x >> 16), static_cast<int>(b.y & 0xffffu), static_cast<int>(b.y >> 16)};
                uint32_t th = 0, ab = 0;
                unsigned long long sq = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    th += static_cast<uint32_t>(abs(ctv[j] - cpv[j]));
                    get[j] += ctv[j];
                    gep[j] += cpv[j];
                    const int d = get[j] - gep[j];
                    ab += static_cast<uint32_t>(abs(d));
                    sq += static_cast<unsigned long long>(static_cast<long long>(d) * d);
                }
                th = __reduce_add_sync(0xffffffffu, th);
                if (lane == 0 && th && prm.thick != nullptr)
                    atomicAdd(reinterpret_cast<unsigned long long*>(prm.thick) + item * K + c, static_cast<unsigned long long>(th));
                if (c >= 1) {                                               // threshold k = c
                    ab = __reduce_add_sync(0xffffffffu, ab);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
                    if (lane == 0 && ab) {                                  // ab == 0 <=> sq == 0
                        if (prm.babs != nullptr) atomicAdd(reinterpret_cast<unsigned long long*>(prm.babs) + item * nthr + (c - 1), static_cast<unsigned long long>(ab));
                        if (prm.bsq != nullptr) atomicAdd(reinterpret_cast<unsigned long long*>(prm.bsq) + item * nthr + (c - 1), sq);
                    }
                    if (valid && prm.bnd_t != nullptr) {
                        const long long o = (item * nthr + (c - 1)) * static_cast<long long>(W) + x;
                        *reinterpret_cast<int4*>(prm.bnd_t + o) = make_int4(H - get[0], H - get[1], H - get[2], H - get[3]);
                        *reinterpret_cast<int4*>(prm.bnd_p + o) = make_int4(H - gep[0], H - gep[1], H - gep[2], H - gep[3]);
                    }
                }
            }
        }
        if (prm.counts != nullptr) {
#pragma unroll 1
            for (int i = lane; i < 256; i += 32) {
                const uint32_t v = counts[i];
                const int t = i >> 4, p = i & 15;
                if (v && t < K && p < K) atomicAdd(prm.counts + item * K * K + t * K + p, static_cast<unsigned long long>(v));
            }
        }
        if (prm.first_pos != nullptr) {
            // lane l ends up with the minimum over the lanes of row l = map * K + class
            uint32_t mine = OCTM_NO_SEED;
#pragma unroll 1
            for (int r = 0; r < 2 * K; ++r) {
                const uint32_t v = __reduce_min_sync(0xffffffffu, fst[r * 32]);
                if (lane == r) mine = v;
            }
            if (lane < 2 * K && mine != OCTM_NO_SEED) atomicMin(prm.first_pos + item * 2 * K + lane, mine);
        }
        if (prm.unsorted != nullptr) {
            uns = __reduce_or_sync(0xffffffffu, uns);
            if (lane == 0 && uns) atomicOr(prm.unsorted + item, uns);
        }
        __syncwarp();
    }
}

// Seeds of the maps the certificate rejected: first raster position of every class by a scan of the labels (K <= 8,
// item_elems % 16 == 0, 16-byte aligned maps: the shapes of the strip kernel).  One CTA per flagged (item, map); a thread
// takes every 256th 16-byte group, in raster order, so a class it has met once can be ignored from then on -- and once it
// has met all K classes it is done (uniform random maps end after a few groups).
__global__ void __launch_bounds__(256) first_pos_fix_kernel(const uint8_t* __restrict__ yt, const uint8_t* __restrict__ yp,
                                                            long long n_items, long long item_elems, int K,
                                                            const uint32_t* __restrict__ unsorted, uint32_t* first_pos) {
    __shared__ uint32_t s_first[8];
    const uint32_t all = (1u << K) - 1u;
    for (long long job = blockIdx.x; job < n_items * 2; job += gridDim.x) {
        const long long item = job >> 1;
        const int m = static_cast<int>(job & 1);
        if (!((unsorted[item] >> m) & 1u)) continue;                  // CTA-uniform
        __syncthreads();
        if (threadIdx.x < 8) s_first[threadIdx.x] = OCTM_NO_SEED;
        __syncthreads();
        const uint4* L = reinterpret_cast<const uint4*>((m ? yp : yt) + item * item_elems);
        const long long groups = item_elems >> 4;
        uint32_t seen = 0;
        auto take = [&](const uint4& w, long long g) {
            // one-hot byte per label: two words share a PRMT selector (their labels in alternate nibbles)
            const uint32_t x0 = (w.x & 0x0f0f0f0fu) | ((w.y & 0x0f0f0f0fu) << 4), x1 = (w.z & 0x0f0f0f0fu) | ((w.w & 0x0f0f0f0fu) << 4);
            const uint32_t lo = 0x08040201u, hi = 0x80402010u;
            uint32_t bits = (prmt(lo, hi, x0) | prmt(lo, hi, x0 >> 16)) | (prmt(lo, hi, x1) | prmt(lo, hi, x1 >> 16));
            bits = (bits | (bits >> 16));
            bits = (bits | (bits >> 8)) & 0xffu;
            uint32_t fresh = bits & ~seen & all;
            seen |= bits;
            while (fresh) {                                   // rare (a class is fresh once per thread and item)
                const int c = __ffs(fresh) - 1;
                fresh &= fresh - 1;
                const uint32_t c4 = 0x01010101u * static_cast<uint32_t>(c);
                auto zb = [&](uint32_t word) -> uint32_t {      // exact zero-byte test of word ^ c4
                    const uint32_t x = word ^ c4;
                    return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
                };
                const uint32_t z0 = zb(w.x), z1 = zb(w.y), z2 = zb(w.z), z3 = zb(w.w);
                const uint32_t pos = z0 ? (__ffs(z0) - 1) >> 3 : (z1 ? 4 + ((__ffs(z1) - 1) >> 3) : (z2 ? 8 + ((__ffs(z2) - 1) >> 3) : 12 + ((__ffs(z3) - 1) >> 3)));
                atomicMin(&s_first[c], static_cast<uint32_t>(g * 16 + pos));
            }
        };
        long long g = threadIdx.x;
        for (; g + 3 * 256 < groups && seen != all; g += 4 * 256) {     // four loads in flight per thread, taken in raster order
            const uint4 w0 = __ldg(L + g), w1 = __ldg(L + g + 256), w2 = __ldg(L + g + 512), w3 = __ldg(L + g + 768);
            take(w0, g);
            take(w1, g + 256);
            take(w2, g + 512);
            take(w3, g + 768);
        }
        for (; g < groups && seen != all; g += 256) take(__ldg(L + g), g);
        __syncthreads();
        if (threadIdx.x < K) first_pos[(item * 2 + m) * K + threadIdx.x] = s_first[threadIdx.x];
    }
}

// Confusion matrices of the items whose two maps the certificate accepted, from their boundary rows b_k(x) = #{label < k}
// alone.  In a column in class order the pixels of class < a form a prefix of length b_a, so
//   C(a, b) = sum_x min(bt_a(x), bp_b(x)) = #{t < a, p < b}   (b_0 = 0, b_K = H)
//   count(t = i, p = j) = C(i+1, j+1) - C(i, j+1) - C(i+1, j) + C(i, j).
// A warp per item (persistent), a lane per 4 columns at a time (16-byte loads of the K-1 rows of each map); the 49 sums
// C(a, b), a, b = 1..7, and the 2 x 7 row sums live in registers and meet in warp reductions.  Rows k >= K are taken as
// b_k = H, which makes the K = 8 arithmetic serve every K.  Items with a rejected map or a label >= K (unsorted != 0) are
// left to confusion_fix_kernel.
constexpr int kRowsWarps = 8;
__global__ void __launch_bounds__(kRowsWarps * 32) confusion_from_rows_kernel(const int* __restrict__ bnd_t, const int* __restrict__ bnd_p,
                                                                              long long n_items, int H, int W, int K,
                                                                              const uint32_t* __restrict__ unsorted,
                                                                              unsigned long long* counts) {
    const int lane = threadIdx.x & 31;
    const long long stride = static_cast<long long>(gridDim.x) * kRowsWarps;
    for (long long item = static_cast<long long>(blockIdx.x) * kRowsWarps + (threadIdx.x >> 5); item < n_items; item += stride) {
        if (unsorted[item] != 0u) continue;                                   // warp-uniform
        uint32_t C[7][7], St[7], Sp[7];
#pragma unroll
        for (int a = 0; a < 7; ++a) {
            St[a] = Sp[a] = 0;
#pragma unroll
            for (int b = 0; b < 7; ++b) C[a][b] = 0;
        }
        const int4* rt = reinterpret_cast<const int4*>(bnd_t + item * (K - 1) * static_cast<long long>(W));
        const int4* rp = reinterpret_cast<const int4*>(bnd_p + item * (K - 1) * static_cast<long long>(W));
        const int W4 = W >> 2;
        for (int q = lane; q < W4; q += 32) {
            int4 t[7], p[7];
#pragma unroll
            for (int a = 0; a < 7; ++a) {
                t[a] = a < K - 1 ? __ldg(rt + a * W4 + q) : make_int4(H, H, H, H);
                p[a] = a < K - 1 ? __ldg(rp + a * W4 + q) : make_int4(H, H, H, H);
            }
#pragma unroll
            for (int a = 0; a < 7; ++a) {
                St[a] += static_cast<uint32_t>(t[a].x + t[a].y + t[a].z + t[a].w);
                Sp[a] += static_cast<uint32_t>(p[a].x + p[a].y + p[a].z + p[a].w);
#pragma unroll
                for (int b = 0; b < 7; ++b)
                    C[a][b] += static_cast<uint32_t>((min(t[a].x, p[b].x) + min(t[a].y, p[b].y)) +
                                                     (min(t[a].z, p[b].z) + min(t[a].w, p[b].w)));
            }
        }
#pragma unroll
        for (int a = 0; a < 7; ++a) {
            St[a] = __reduce_add_sync(0xffffffffu, St[a]);
            Sp[a] = __reduce_add_sync(0xffffffffu, Sp[a]);
#pragma unroll
            for (int b = 0; b < 7; ++b) C[a][b] = __reduce_add_sync(0xffffffffu, C[a][b]);
        }
        // C(a, b) over a, b = 0..8 (index 8: b_8 = H; with K < 8 the rows from K on are H already)
        const uint32_t HW = static_cast<uint32_t>(H) * static_cast<uint32_t>(W);
        auto cab = [&](int a, int b) -> uint32_t {
            if (a == 0 || b == 0) return 0u;
            if (a == 8 && b == 8) return HW;
            if (a == 8) return Sp[b - 1];
            if (b == 8) return St[a - 1];
            return C[a - 1][b - 1];
        };
        unsigned long long* out = counts + item * K * K;
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t v = cab(i + 1, j + 1) - cab(i, j + 1) - cab(i + 1, j) + cab(i, j);
                if (i < K && j < K && lane == ((i * 8 + j) & 31)) out[i * K + j] = v;
            }
    }
}

// Confusion matrices of the items confusion_from_rows_kernel leaves (a map the certificate rejected, or a label >= K):
// the per-pixel histogram (K <= 8, W % 16 == 0, 16-byte aligned maps: the shapes of the strip kernel), with the strip
// kernel's treatment of bad labels: a 128-column strip of the item that holds a label >= 8 contributes nothing (its warp
// withholds its counts there), codes with a label in [K, 8) are dropped at the output.  Either way the item's counts fall
// short of H * W.  One CTA per such item (grid-stride, one CTA-uniform skip per item as in first_pos_fix_kernel); a
// thread takes every 256th 16-byte group of both maps, and a group of one joint code adds 16 at once.  Items with a label
// >= K (the transient bit kBadLabels, cleared here) are read twice: once for the strips to leave out.
__global__ void __launch_bounds__(256) confusion_fix_kernel(const uint8_t* __restrict__ yt, const uint8_t* __restrict__ yp,
                                                            long long n_items, int H, int W, int K, uint32_t* unsorted,
                                                            unsigned long long* counts) {
    __shared__ uint32_t s_hist[8][64][16];      // u16 [warp][code t*8+p][lane]: at most H * W / 256 <= 2^15 per lane
    __shared__ uint32_t s_sum[64];
    __shared__ uint32_t s_bad_strips;           // bit s: strip s (columns 128 s ..) holds a label >= 8 (W <= 2048)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < 8 * 64 * 16; i += 256) (&s_hist[0][0][0])[i] = 0;
    __syncthreads();
    unsigned short* hist_lane = reinterpret_cast<unsigned short*>(&s_hist[warp][0][0]) + lane;
    const long long item_elems = static_cast<long long>(H) * W;
    const int groups = static_cast<int>(item_elems >> 4), row_groups = W >> 4;     // H * W <= 2^23
    for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
        const uint32_t u = unsorted[item];
        if (u == 0u) continue;                                                // CTA-uniform: counted from the rows
        if (tid < 64) s_sum[tid] = 0;
        if (tid == 0) s_bad_strips = 0;
        const uint4* T = reinterpret_cast<const uint4*>(yt + item * item_elems);
        const uint4* P = reinterpret_cast<const uint4*>(yp + item * item_elems);
        __syncthreads();
        uint32_t bad_strips = 0;
        if (u & kBadLabels) {                                                 // CTA-uniform, rare
            uint32_t mine = 0;
            for (int g = tid; g < groups; g += 256) {
                const uint4 a = __ldg(T + g), b = __ldg(P + g);
                if ((((a.x | a.y) | (a.z | a.w)) | ((b.x | b.y) | (b.z | b.w))) & 0xf8f8f8f8u)
                    mine |= 1u << ((g % row_groups) >> 3);
            }
            mine = __reduce_or_sync(0xffffffffu, mine);
            if (lane == 0 && mine) atomicOr(&s_bad_strips, mine);
            __syncthreads();
            bad_strips = s_bad_strips;
        }
        for (int g = tid; g < groups; g += 256) {
            if (bad_strips && ((bad_strips >> ((g % row_groups) >> 3)) & 1u)) continue;
            const uint4 a = __ldg(T + g), b = __ldg(P + g);                   // labels < 8 from here on
            const uint32_t j[4] = {a.x * 8u + b.x, a.y * 8u + b.y, a.z * 8u + b.z, a.w * 8u + b.w};
            const uint32_t c = prmt(j[0], 0, 0);
            if ((((j[0] ^ c) | (j[1] ^ c)) | ((j[2] ^ c) | (j[3] ^ c))) == 0u) {
                hist_add(hist_lane, c & 0x3fu, 16);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int i = 0; i < 4; ++i) hist_add(hist_lane, (j[k] >> (8 * i)) & 0x3fu, 1);
            }
        }
        __syncthreads();
        {
            // code c = tid % 64 over the lanes of warps 2 q and 2 q + 1, q = tid / 64; the rotation spreads the banks
            const int c = tid & 63, q = tid >> 6;
            uint32_t sum = 0;
#pragma unroll
            for (int w = 0; w < 2; ++w)
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    uint32_t& h = s_hist[2 * q + w][c][(c + i) & 15];
                    sum += (h & 0xffffu) + (h >> 16);
                    h = 0;
                }
            atomicAdd(&s_sum[c], sum);
        }
        __syncthreads();
        for (int i = tid; i < K * K; i += 256) counts[item * K * K + i] = s_sum[(i / K) * 8 + i % K];
        if (tid == 0) unsorted[item] = u & 3u;
        __syncthreads();
    }
}

// K3: sums over columns of (bt - bp)^2 and |bt - bp| for int32 boundary arrays [n][Kb][W].
__global__ void __launch_bounds__(256) boundary_error_kernel(const int* __restrict__ bt, const int* __restrict__ bp,
                                                             long long n_rows, int W, long long* sum_sq,
                                                             long long* sum_abs) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = static_cast<long long>(blockIdx.x) * 8 + warp;
    if (row >= n_rows) return;
    const int* a = bt + row * W;
    const int* b = bp + row * W;
    long long sq = 0, ab = 0;
    for (int x = lane; x < W; x += 32) {
        const long long d = static_cast<long long>(a[x]) - b[x];
        sq += d * d;
        ab += d < 0 ? -d : d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        ab += __shfl_xor_sync(0xffffffffu, ab, o);
    }
    if (lane == 0) {
        sum_sq[row] = sq;
        sum_abs[row] = ab;
    }
}

__global__ void __launch_bounds__(256) max_label_kernel(const uint8_t* __restrict__ x, long long n, uint32_t* out) {
    uint32_t m = 0;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) m = max(m, (uint32_t)x[i]);
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// ------------------------------------------------------------------------------------ dispatch
static bool fast_ok(int H, int W, int K, const void* a, const void* b) {
    return K >= 2 && K <= 8 && W % 16 == 0 && W >= 16 && W <= 2048 && H >= 1 && H <= 4096 &&
           (reinterpret_cast<uintptr_t>(a) % 16 == 0) && (reinterpret_cast<uintptr_t>(b) % 16 == 0);
}

// cuTensorMapEncodeTiled, fetched through the runtime so that liboctm.so does not link libcuda
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}

// label tensor [n_items * H rows][W columns] of uint8; one box = R rows x min(W, 128) columns, dense in smem
static int make_label_map(CUtensorMap* tm, const uint8_t* base, long long rows, int W, int R) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (enc == nullptr) return fail(OCTM_ERR_LAUNCH, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(rows)};
    const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(W)};            // bytes between rows
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(W < kStrip ? W : kStrip), static_cast<cuuint32_t>(R)};
    const cuuint32_t estride[2] = {1, 1};
    const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(base), gdim, gstride, box, estride,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(OCTM_ERR_LAUNCH, "cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r));
    return OCTM_OK;
}

template <int NP, bool CONF, bool COLS, bool SEEDS, bool SORT>
static int launch_fast(const LabelPassParams& p0, cudaStream_t stream) {
    LabelPassParams p = p0;
    p.one = 1;
    const int NW = (p.W + kStrip - 1) / kStrip;
    // each warp stages its own 128-column strip: R rows per stage (multiple of 4), S stages.  16 rows x 2 stages =
    // 8 KB of ring per warp; shared memory (occupancy) matters more than ring depth here.
    const int R = 16, S = 2;
    p.R = R;
    p.S = S;
    const int srow = p.W < kStrip ? p.W : kStrip;
    const int state = kWarpBars + (p.H > kShortRows ? kWarpBytesTall : kWarpBytesShort);
    const int stage = 2 * R * srow;
    const int budget = max_optin_smem();
    const int smem = kOffWarp + NW * (state + S * stage);
    if (smem > budget) return fail(OCTM_ERR_UNSUPPORTED, "label pass: %d B of shared memory needed", smem);
    // the warps of a CTA merge their strips in the outputs by global reductions: start from zero / "no seed"
    {
        const size_t n = static_cast<size_t>(p.n_items), k = static_cast<size_t>(p.K);
        bool ok = true;
        if (p.counts) ok = ok && cudaMemsetAsync(p.counts, 0, n * k * k * 8, stream) == cudaSuccess;
        if (p.thick) ok = ok && cudaMemsetAsync(p.thick, 0, n * k * 8, stream) == cudaSuccess;
        if (p.bsq) ok = ok && cudaMemsetAsync(p.bsq, 0, n * (k - 1) * 8, stream) == cudaSuccess;
        if (p.babs) ok = ok && cudaMemsetAsync(p.babs, 0, n * (k - 1) * 8, stream) == cudaSuccess;
        if (p.first_pos) ok = ok && cudaMemsetAsync(p.first_pos, 0xff, n * 2 * k * 4, stream) == cudaSuccess;
        if (p.unsorted) ok = ok && cudaMemsetAsync(p.unsorted, 0, n * 4, stream) == cudaSuccess;
        if (!ok) return fail(OCTM_ERR_LAUNCH, "label pass: clearing the outputs failed");
    }
    CUtensorMap tm_true, tm_pred;
    const long long rows = p.n_items * p.H;
    if (int e = make_label_map(&tm_true, p.yt, rows, p.W, R)) return e;
    if (int e = make_label_map(&tm_pred, p.yp, rows, p.W, R)) return e;
    auto kern = NW > 8 ? label_pass_fast<NP, CONF, COLS, SEEDS, SORT, true> : label_pass_fast<NP, CONF, COLS, SEEDS, SORT, false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, budget) != cudaSuccess)
        return fail(OCTM_ERR_LAUNCH, "cudaFuncSetAttribute(label_pass_fast) failed");
    const int threads = NW * 32;
    const long long grid = resident_grid(p.n_items, kern, threads, smem, 1);      // persistent: the CTAs resident at once
    OCTM_TIMED("label_pass_fast", stream) kern<<<static_cast<unsigned>(grid), threads, smem, stream>>>(p, tm_true, tm_pred);
    if (int e = check_launch("label_pass_fast")) return e;
    if (SORT && !SEEDS && p.first_pos != nullptr) {
        long long fgrid = p.n_items * 2;
        const long long fcap = static_cast<long long>(sm_count()) * 8;
        if (fgrid > fcap) fgrid = fcap;
        OCTM_TIMED("first_pos_fix_kernel", stream) first_pos_fix_kernel<<<static_cast<unsigned>(fgrid), 256, 0, stream>>>(
            p.yt, p.yp, p.n_items, static_cast<long long>(p.H) * p.W, p.K, p.unsorted, p.first_pos);
        return check_launch("first_pos_fix_kernel");
    }
    return OCTM_OK;
}

template <bool CONF, bool COLS, bool SEEDS, bool SORT>
static int dispatch_np(const LabelPassParams& p, cudaStream_t stream) {
    const int np = p.K / 2;   // ceil((K-1)/2)
    switch (np) {
        case 1: return launch_fast<1, CONF, COLS, SEEDS, SORT>(p, stream);
        case 2: return launch_fast<2, CONF, COLS, SEEDS, SORT>(p, stream);
        case 3: return launch_fast<3, CONF, COLS, SEEDS, SORT>(p, stream);
        default: return launch_fast<4, CONF, COLS, SEEDS, SORT>(p, stream);
    }
}

static int launch_generic(const LabelPassParams& p, cudaStream_t stream) {
    // K <= 16 with 4-byte rows: the warp-per-strip kernel; anything else the byte-wise one
    const bool wide = p.W % 4 == 0 && reinterpret_cast<uintptr_t>(p.yt) % 4 == 0 && reinterpret_cast<uintptr_t>(p.yp) % 4 == 0 &&
                      (p.bnd_t == nullptr || (reinterpret_cast<uintptr_t>(p.bnd_t) % 16 == 0 && reinterpret_cast<uintptr_t>(p.bnd_p) % 16 == 0)) &&
                      p.H <= 16383 && static_cast<long long>(p.H) * p.W < (1ll << 32) &&
                      // a handful of items (one volume) is latency-bound either way: the byte-wise kernel's 32-column warps
                      // then give four times as many walkers (cfg2, 49 items: 0.09 against 0.21 ms)
                      p.n_items * ((p.W + 127) / 128) >= 2ll * sm_count() * kWideWarps;
    // few items: one CTA per 256-column strip, partial results joined by atomics on zero-initialised outputs
    const long long resident = static_cast<long long>(sm_count()) * 8;
    const int strips = wide ? (p.W + 127) / 128 : (p.n_items < resident && p.W > 256 ? (p.W + 255) / 256 : 1);
    if (wide || strips > 1) {
        const size_t n = static_cast<size_t>(p.n_items), k = static_cast<size_t>(p.K);
        bool ok = true;
        if (p.counts) ok = ok && cudaMemsetAsync(p.counts, 0, n * k * k * 8, stream) == cudaSuccess;
        if (p.thick) ok = ok && cudaMemsetAsync(p.thick, 0, n * k * 8, stream) == cudaSuccess;
        if (p.bsq) ok = ok && cudaMemsetAsync(p.bsq, 0, n * (k - 1) * 8, stream) == cudaSuccess;
        if (p.babs) ok = ok && cudaMemsetAsync(p.babs, 0, n * (k - 1) * 8, stream) == cudaSuccess;
        if (p.first_pos) ok = ok && cudaMemsetAsync(p.first_pos, 0xff, n * 2 * k * 4, stream) == cudaSuccess;
        if (!ok) return fail(OCTM_ERR_LAUNCH, "memset of the label-pass outputs failed");
    }
    if (p.unsorted != nullptr && cudaMemsetAsync(p.unsorted, 0, static_cast<size_t>(p.n_items) * 4, stream) != cudaSuccess)
        return fail(OCTM_ERR_LAUNCH, "memset of the label-pass outputs failed");
    if (wide) {
        const int kWideSmem = kWideWarps * wide_warp_bytes(p.K);
        if (cudaFuncSetAttribute(label_pass_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, kWideWarps * wide_warp_bytes(16)) != cudaSuccess)
            return fail(OCTM_ERR_LAUNCH, "cudaFuncSetAttribute(label_pass_wide) failed");
        const long long grid = resident_grid((p.n_items * strips + kWideWarps - 1) / kWideWarps, label_pass_wide, kWideWarps * 32,
                                             kWideSmem, 3);
        OCTM_TIMED("label_pass_wide", stream) label_pass_wide<<<static_cast<unsigned>(grid), kWideWarps * 32, kWideSmem, stream>>>(p, strips);
        return check_launch("label_pass_wide");
    }
    long long grid = p.n_items * strips;
    if (grid > resident) grid = resident;
    OCTM_TIMED("label_pass_generic", stream) label_pass_generic<<<static_cast<unsigned>(grid), 256, 0, stream>>>(p, strips);
    return check_launch("label_pass_generic");
}

// ------------------------------------------------------------------------------------ where the seeds come from
// With the certificate the strip kernel has two ways to the contour seeds: from the column totals in the item epilogue
// (free, but the maps the certificate rejects are rescanned by first_pos_fix_kernel: 0.95 ms per 16,384 rejected maps),
// or tracked per pixel (+0.35 ms per 16,384 items whatever the data).  Clean data wants the first, a stream of
// predictions that are mostly out of class order (any real argmax) the second.  The choice follows the data: every call
// leaves "maps rejected / maps seen" in a host-mapped word (one tiny kernel, no synchronisation: the next call reads
// whatever has arrived), and a call tracks per pixel when more than a fifth of the maps of the last report were
// rejected.  Both ways give the same seeds (tests run both); octm_label_pass_seed_policy pins one.
// The confusion matrices follow the same choice.  On a mostly accepted stream the strip kernel runs without its per-pixel
// histogram, and the counts come from the boundary rows (confusion_from_rows_kernel) plus a per-pixel histogram of just
// the rejected items (confusion_fix_kernel).  On a mostly rejected stream that would read the labels twice, so the strip
// kernel keeps its histogram.
// The report: host_report(kReportSeeds), [0] rejected maps, [1] maps.
static std::atomic<int> g_seed_policy{0};      // 0 follow the data, 1 column totals + rescans, 2 per pixel

__global__ void __launch_bounds__(1024) seed_feedback_kernel(const uint32_t* __restrict__ unsorted, long long n, uint32_t* out) {
    __shared__ uint32_t s_sum[32];
    uint32_t c = 0;
    for (long long i = threadIdx.x; i < n; i += 1024) c += __popc(unsorted[i] & 3u);
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x < 32) {
        c = __reduce_add_sync(0xffffffffu, s_sum[threadIdx.x]);
        if (threadIdx.x == 0) {
            out[1] = static_cast<uint32_t>(min(2 * n, static_cast<long long>(0xffffffffu)));
            out[0] = c;
        }
    }
}

bool stream_mostly_rejected() {
    const int policy = g_seed_policy.load();
    if (policy != 0) return policy == 2;
    HostReport* f = host_report(kReportSeeds);
    if (f == nullptr) return false;
    const uint32_t rejected = *static_cast<volatile uint32_t*>(f->host), maps = *static_cast<volatile uint32_t*>(f->host + 1);
    return maps != 0 && static_cast<unsigned long long>(rejected) * 5ull > maps;
}

static int report_rejected(const LabelPassParams& p, cudaStream_t stream) {
    HostReport* f = host_report(kReportSeeds);
    if (f == nullptr) return OCTM_OK;
    OCTM_TIMED("seed_feedback_kernel", stream) seed_feedback_kernel<<<1, 1024, 0, stream>>>(p.unsorted, p.n_items, f->dev);
    return check_launch("seed_feedback_kernel");
}

// counts of a certified strip-kernel pass that ran without its histogram: accepted items from their boundary rows,
// the others pixel by pixel (every item's K x K counts are written by exactly one of the two kernels)
static int confusion_from_rows(const LabelPassParams& p, cudaStream_t stream) {
    const long long rgrid = resident_grid((p.n_items + kRowsWarps - 1) / kRowsWarps, confusion_from_rows_kernel, kRowsWarps * 32, 0, 2);
    OCTM_TIMED("confusion_from_rows_kernel", stream) confusion_from_rows_kernel<<<static_cast<unsigned>(rgrid), kRowsWarps * 32, 0, stream>>>(
        p.bnd_t, p.bnd_p, p.n_items, p.H, p.W, p.K, p.unsorted, p.counts);
    if (int e = check_launch("confusion_from_rows_kernel")) return e;
    const long long fgrid = resident_grid(p.n_items, confusion_fix_kernel, 256, 0, 4);
    OCTM_TIMED("confusion_fix_kernel", stream) confusion_fix_kernel<<<static_cast<unsigned>(fgrid), 256, 0, stream>>>(
        p.yt, p.yp, p.n_items, p.H, p.W, p.K, p.unsorted, p.counts);
    return check_launch("confusion_fix_kernel");
}

int run_label_pass(const LabelPassParams& p, bool conf, bool cols, bool seeds, cudaStream_t stream) {
    if (p.n_items == 0) return OCTM_OK;
    if (fast_ok(p.H, p.W, p.K, p.yt, p.yp) && p.n_items * p.H < (1ll << 31) /* TMA row coordinate */ &&
        (p.bnd_t == nullptr || reinterpret_cast<uintptr_t>(p.bnd_t) % 16 == 0) &&
        (p.bnd_p == nullptr || reinterpret_cast<uintptr_t>(p.bnd_p) % 16 == 0)) {
        // the suite's call: certificate; seeds (if asked for) from the column totals, rescanned for rejected maps
        if (p.unsorted != nullptr) {
            const bool per_pixel = stream_mostly_rejected();
            int e;
            if (!per_pixel && p.bnd_t != nullptr) {
                LabelPassParams q = p;
                q.counts = nullptr;                  // written whole by the two kernels below
                e = dispatch_np<false, true, false, true>(q, stream);
                if (e == OCTM_OK) e = confusion_from_rows(p, stream);
            } else {
                e = p.first_pos != nullptr && per_pixel ? dispatch_np<true, true, true, true>(p, stream)
                                                        : dispatch_np<true, true, false, true>(p, stream);
            }
            if (e != OCTM_OK) return e;
            return report_rejected(p, stream);
        }
        if (conf && cols && seeds) return dispatch_np<true, true, true, false>(p, stream);
        if (conf && cols) return dispatch_np<true, true, false, false>(p, stream);
        if (conf && !cols && !seeds) return dispatch_np<true, false, false, false>(p, stream);
        if (!conf && cols && !seeds) return dispatch_np<false, true, false, false>(p, stream);
        return dispatch_np<true, true, true, false>(p, stream);
    }
    return launch_generic(p, stream);
}

}  // namespace octm

using octm::LabelPassParams;

static int check_common(const void* yt, const void* yp, int64_t n, int K) {
    if (n < 0) return octm::fail(OCTM_ERR_INVALID, "n_items < 0");
    if (K < 2 || K > OCTM_MAX_CLASSES) return octm::fail(OCTM_ERR_INVALID, "num_classes %d outside [2, 16]", K);
    if (n > 0 && (yt == nullptr || yp == nullptr)) return octm::fail(OCTM_ERR_INVALID, "null label pointer");
    return OCTM_OK;
}

extern "C" int octm_label_pass_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                  int num_classes, uint64_t* counts, int64_t* thick_absdiff, int64_t* bnd_sq,
                                  int64_t* bnd_abs, int32_t* bnd_true, int32_t* bnd_pred, uint32_t* first_pos,
                                  void* stream) {
    return octm_label_pass_sorted_u8(y_true, y_pred, n_items, H, W, num_classes, counts, thick_absdiff, bnd_sq, bnd_abs,
                                     bnd_true, bnd_pred, first_pos, nullptr, stream);
}

extern "C" int octm_label_pass_sorted_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                         int num_classes, uint64_t* counts, int64_t* thick_absdiff, int64_t* bnd_sq,
                                         int64_t* bnd_abs, int32_t* bnd_true, int32_t* bnd_pred, uint32_t* first_pos,
                                         uint32_t* unsorted, void* stream) {
    if (int e = check_common(y_true, y_pred, n_items, num_classes)) return e;
    if (H < 1 || W < 1) return octm::fail(OCTM_ERR_INVALID, "H, W must be >= 1");
    if (static_cast<long long>(H) * W >= (1ll << 32)) return octm::fail(OCTM_ERR_UNSUPPORTED, "H*W >= 2^32");
    if ((bnd_true == nullptr) != (bnd_pred == nullptr)) return octm::fail(OCTM_ERR_INVALID, "bnd_true/bnd_pred: both or neither");
    LabelPassParams p{};
    p.yt = y_true; p.yp = y_pred; p.n_items = n_items; p.H = H; p.W = W; p.K = num_classes;
    p.counts = reinterpret_cast<unsigned long long*>(counts);
    p.thick = reinterpret_cast<long long*>(thick_absdiff);
    p.bsq = reinterpret_cast<long long*>(bnd_sq);
    p.babs = reinterpret_cast<long long*>(bnd_abs);
    p.bnd_t = bnd_true; p.bnd_p = bnd_pred; p.first_pos = first_pos; p.unsorted = unsorted;
    if (unsorted != nullptr && !(counts && thick_absdiff && bnd_sq && bnd_abs))
        return octm::fail(OCTM_ERR_INVALID, "unsorted needs counts and the column sums");
    const bool conf = counts != nullptr;
    const bool cols = thick_absdiff || bnd_sq || bnd_abs || bnd_true;
    const bool seeds = first_pos != nullptr;
    return octm::run_label_pass(p, conf, cols, seeds, static_cast<cudaStream_t>(stream));
}

extern "C" int octm_label_pass_seed_policy(int policy) {
    if (policy < 0 || policy > 2) return octm::g_seed_policy.load();
    return octm::g_seed_policy.exchange(policy);
}

extern "C" int octm_label_pass_path(int H, int W, int num_classes, const void* y_true, const void* y_pred) {
    if (octm::fast_ok(H, W, num_classes, y_true, y_pred)) return 1;
    return W % 4 == 0 && reinterpret_cast<uintptr_t>(y_true) % 4 == 0 && reinterpret_cast<uintptr_t>(y_pred) % 4 == 0 && H <= 16383 &&
                   static_cast<long long>(H) * W < (1ll << 32)
               ? 2
               : 0;
}

extern "C" int octm_confusion_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int64_t item_elems,
                                 int num_classes, uint64_t* counts, void* stream) {
    if (int e = check_common(y_true, y_pred, n_items, num_classes)) return e;
    if (counts == nullptr) return octm::fail(OCTM_ERR_INVALID, "counts is null");
    if (item_elems < 1 || item_elems >= (1ll << 32)) return octm::fail(OCTM_ERR_INVALID, "item_elems outside [1, 2^32)");
    // any factorisation H*W = item_elems gives the same histogram: prefer one the fast kernel takes
    int H = 1, W = 0;
    for (int w = 2048; w >= 16; w >>= 1) {
        if (item_elems % w == 0 && item_elems / w <= 4096) { W = w; H = static_cast<int>(item_elems / w); break; }
    }
    if (W == 0) {
        if (item_elems > 0x7fffffff) return octm::fail(OCTM_ERR_UNSUPPORTED, "item too large for the generic kernel");
        W = static_cast<int>(item_elems); H = 1;
        // generic kernel walks columns: make rows long-ish
        for (int h = 64; h >= 2; --h) if (item_elems % h == 0) { H = h; W = static_cast<int>(item_elems / h); break; }
    }
    LabelPassParams p{};
    p.yt = y_true; p.yp = y_pred; p.n_items = n_items; p.H = H; p.W = W; p.K = num_classes;
    p.counts = reinterpret_cast<unsigned long long*>(counts);
    return octm::run_label_pass(p, true, false, false, static_cast<cudaStream_t>(stream));
}

extern "C" int octm_column_scan_u8(const uint8_t* y_true, const uint8_t* y_pred, int64_t n_items, int H, int W,
                                   int num_classes, int64_t* thick_absdiff, int64_t* bnd_sq, int64_t* bnd_abs,
                                   int32_t* bnd_true, int32_t* bnd_pred, void* stream) {
    return octm_label_pass_u8(y_true, y_pred, n_items, H, W, num_classes, nullptr, thick_absdiff, bnd_sq, bnd_abs,
                              bnd_true, bnd_pred, nullptr, stream);
}

extern "C" int octm_boundary_error_i32(const int32_t* bnd_true, const int32_t* bnd_pred, int64_t n_items,
                                       int num_boundaries, int W, int64_t* sum_sq, int64_t* sum_abs, void* stream) {
    if (n_items < 0 || num_boundaries < 1 || W < 1) return octm::fail(OCTM_ERR_INVALID, "bad shape");
    if (n_items == 0) return OCTM_OK;
    if (!bnd_true || !bnd_pred || !sum_sq || !sum_abs) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    const long long rows = n_items * num_boundaries;
    OCTM_TIMED("boundary_error_kernel", static_cast<cudaStream_t>(stream)) octm::boundary_error_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        bnd_true, bnd_pred, rows, W, reinterpret_cast<long long*>(sum_sq), reinterpret_cast<long long*>(sum_abs));
    return octm::check_launch("boundary_error_kernel");
}

extern "C" int octm_validate_labels_u8(const uint8_t* labels, int64_t n_elems, uint32_t* max_label, void* stream) {
    if (n_elems < 0 || max_label == nullptr || (n_elems > 0 && labels == nullptr)) return octm::fail(OCTM_ERR_INVALID, "bad argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (cudaMemsetAsync(max_label, 0, sizeof(uint32_t), s) != cudaSuccess) return octm::fail(OCTM_ERR_LAUNCH, "memset failed");
    if (n_elems == 0) return OCTM_OK;
    OCTM_TIMED("max_label_kernel", s) octm::max_label_kernel<<<148 * 8, 256, 0, s>>>(labels, n_elems, max_label);
    return octm::check_launch("max_label_kernel");
}
