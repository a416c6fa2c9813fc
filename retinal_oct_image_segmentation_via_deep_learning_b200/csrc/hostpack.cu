// Transfer encoding for host-resident label maps: two labels per byte across PCIe.
//
// The end-to-end path (suite.evaluate_host) is bound by the host->device copy (~50 GB/s on the B200 boxes)
// while the kernels need a tenth of that time.  Labels of a K <= 16 class problem are 4-bit values, so the
// host can pack them in pairs (dst[i] = src[2i] | src[2i+1] << 4, AVX2, all cores), half the bytes cross the
// bus, and a streaming kernel expands them in HBM.  This is a data format conversion, not a metric
// computation: no metric arithmetic runs on the host.  Opt-in (evaluate_host(pack=True)): on the 16-core
// B200 boxes the packer sustains ~80-100 GB/s of input, which merely ties with the plain 50 GB/s copy.
#include <cpuid.h>
#include <immintrin.h>

#include <thread>
#include <vector>

#include "common.cuh"

namespace octm {

// Both packers return the OR of the labels they read: a value >= 16 means that some label has no 4-bit code.
static uint32_t pack_scalar(const uint8_t* src, uint8_t* dst, size_t b, size_t e) {
    uint32_t seen = 0;
    for (size_t i = b; i + 2 <= e; i += 2) {
        seen |= src[i] | src[i + 1];
        dst[i >> 1] = static_cast<uint8_t>((src[i] & 15u) | (src[i + 1] << 4));
    }
    return seen;
}

__attribute__((target("avx2"))) static uint32_t pack_avx2(const uint8_t* src, uint8_t* dst, size_t b, size_t e) {
    size_t i = b;
    const __m256i lo8 = _mm256_set1_epi16(0x00ff);
    __m256i seen = _mm256_setzero_si256();
    const bool aligned = (reinterpret_cast<uintptr_t>(dst + (b >> 1)) & 31u) == 0;
    for (; i + 64 <= e; i += 64) {
        const __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i));
        const __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i + 32));
        seen = _mm256_or_si256(seen, _mm256_or_si256(a, c));
        // per 16-bit lane (even byte, odd byte): even | odd << 4 in the low byte
        __m256i pa = _mm256_and_si256(_mm256_or_si256(a, _mm256_srli_epi16(a, 4)), lo8);
        __m256i pc = _mm256_and_si256(_mm256_or_si256(c, _mm256_srli_epi16(c, 4)), lo8);
        __m256i p = _mm256_permute4x64_epi64(_mm256_packus_epi16(pa, pc), 0xD8);
        if (aligned) _mm256_stream_si256(reinterpret_cast<__m256i*>(dst + (i >> 1)), p);      // written once, read by DMA
        else _mm256_storeu_si256(reinterpret_cast<__m256i*>(dst + (i >> 1)), p);
    }
    const uint32_t tail = pack_scalar(src, dst, i, e);
    _mm_sfence();
    return tail | (_mm256_testz_si256(seen, _mm256_set1_epi8(static_cast<char>(0xf0))) ? 0u : 16u);
}

// 16 packed bytes -> 32 labels
__global__ void __launch_bounds__(256) unpack_nibbles_kernel(const uint4* __restrict__ packed, long long n_vec, uint4* __restrict__ out) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
        const uint4 p = packed[i];
        const uint32_t w[4] = {p.x, p.y, p.z, p.w};
        uint32_t o[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // bytes b0 b1 b2 b3 -> (b0 & 15, b0 >> 4, b1 & 15, b1 >> 4) and the same for b2, b3
            const uint32_t lo = w[k] & 0x0f0f0f0fu, hi = (w[k] >> 4) & 0x0f0f0f0fu;
            o[2 * k] = __byte_perm(lo, hi, 0x5140);
            o[2 * k + 1] = __byte_perm(lo, hi, 0x7362);
        }
        out[2 * i] = make_uint4(o[0], o[1], o[2], o[3]);
        out[2 * i + 1] = make_uint4(o[4], o[5], o[6], o[7]);
    }
}

__global__ void unpack_nibbles_tail_kernel(const uint8_t* __restrict__ packed, long long first, long long n_packed, uint8_t* __restrict__ out,
                                           long long n_out) {
    const long long i = first + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n_packed) {
        const uint32_t b = packed[i];
        out[2 * i] = b & 15u;
        if (2 * i + 1 < n_out) out[2 * i + 1] = b >> 4;
    }
}

}  // namespace octm

extern "C" int octm_host_pack_nibbles(const uint8_t* src, uint8_t* dst, size_t n_labels, int threads) {
    if (n_labels == 0) return OCTM_OK;
    if (!src || !dst) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    if (threads < 1) threads = static_cast<int>(std::thread::hardware_concurrency());
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    static const bool have_avx2 = __builtin_cpu_supports("avx2");
    const size_t even = n_labels & ~static_cast<size_t>(1);
    size_t per = ((even / threads) + 63) & ~static_cast<size_t>(63);
    if (per < (1u << 16)) per = 1u << 16;                      // not worth a thread below 64 KB
    std::vector<uint32_t> seen((even + per - 1) / per + 1, 0u);      // one slot per thread: no shared writes
    auto work = [&](size_t t, size_t b, size_t e) {
        seen[t] = have_avx2 ? octm::pack_avx2(src, dst, b, e) : octm::pack_scalar(src, dst, b, e);
    };
    std::vector<std::thread> pool;
    for (size_t b = per; b < even; b += per) pool.emplace_back(work, b / per, b, b + per < even ? b + per : even);
    work(0, 0, per < even ? per : even);
    for (auto& t : pool) t.join();
    uint32_t any = 0;
    for (uint32_t v : seen) any |= v;
    if (n_labels & 1) {
        any |= src[n_labels - 1];
        dst[n_labels >> 1] = src[n_labels - 1] & 15u;
    }
    return any >= 16u ? OCTM_PACK_WIDE_LABEL : OCTM_OK;
}

extern "C" int octm_unpack_nibbles_u8(const uint8_t* packed, int64_t n_labels, uint8_t* labels, void* stream) {
    if (n_labels < 0) return octm::fail(OCTM_ERR_INVALID, "n_labels < 0");
    if (n_labels == 0) return OCTM_OK;
    if (!packed || !labels) return octm::fail(OCTM_ERR_INVALID, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n_packed = (n_labels + 1) / 2;
    long long n_vec = 0;
    if (reinterpret_cast<uintptr_t>(packed) % 16 == 0 && reinterpret_cast<uintptr_t>(labels) % 16 == 0) n_vec = n_labels / 32;
    if (n_vec > 0) {
        long long blocks = (n_vec + 255) / 256;
        const long long cap = static_cast<long long>(octm::sm_count()) * 8;
        if (blocks > cap) blocks = cap;
        OCTM_TIMED("unpack_nibbles_kernel", st) octm::unpack_nibbles_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(reinterpret_cast<const uint4*>(packed), n_vec,
                                                                                  reinterpret_cast<uint4*>(labels));
        if (int e = octm::check_launch("unpack_nibbles_kernel")) return e;
    }
    const long long first = n_vec * 16;
    if (first < n_packed) {
        const long long rest = n_packed - first;
        OCTM_TIMED("unpack_nibbles_tail_kernel", st) octm::unpack_nibbles_tail_kernel<<<static_cast<unsigned>((rest + 255) / 256), 256, 0, st>>>(packed, first, n_packed, labels, n_labels);
        if (int e = octm::check_launch("unpack_nibbles_tail_kernel")) return e;
    }
    return OCTM_OK;
}
