// skm_common.cuh — shared device helpers for the Snekmer hot-path kernels (sm_100a).
//
// The central piece is warp_scan_sequence(): one warp walks one sequence of the
// packed residue buffer with aligned 32-bit loads (4 residues per lane, 128 per
// warp step), applies the reduction alphabet from a 256-byte shared-memory LUT
// and forms the base-|A| code of the k-mer window starting at every position.
// Neighbouring residues come from the next lanes through warp shuffles, so the
// global buffer is read exactly once, coalesced.  Windows never cross the
// sequence end: positions outside [b, e) carry the invalid symbol, which
// poisons every window covering them — the same rule that makes X/B/Z/*/lower
// case invalid (vectorize.py:239-249 in the reference).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skm_b200.h"

namespace skm {

constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int SYM_INVALID = 0xFF;

// thread-local error string shared by all translation units (skm_api.cu)
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);
int sm_count();

#define SKM_CUDA_TRY(expr)                                        \
    do {                                                          \
        cudaError_t _e = (expr);                                  \
        if (_e != cudaSuccess) return skm::cuda_fail(_e, #expr);  \
    } while (0)

#define SKM_LAUNCH_CHECK(what)                                    \
    do {                                                          \
        cudaError_t _e = cudaGetLastError();                      \
        if (_e != cudaSuccess) return skm::cuda_fail(_e, what);   \
    } while (0)

template <typename T> struct code_traits;
template <> struct code_traits<uint32_t> { static constexpr uint32_t none = 0xFFFFFFFFu; };
template <> struct code_traits<uint64_t> { static constexpr uint64_t none = ~0ull; };

// number of neighbour words a lane needs for k-mers of length k (k-1 residues
// past its own 4): ceil((k-1)/4), rounded up to a supported template value.
inline int neighbour_words(int k) {
    int nw = (k - 1 + 3) / 4;
    if (nw <= 1) return 1;
    if (nw <= 2) return 2;
    if (nw <= 4) return 4;
    if (nw <= 8) return 8;
    return 16;
}
constexpr int SKM_MAX_K = 64;  // 4*16 + 1 would be 65; nsym^k <= 2^64 caps k at 64

// Load the 4 residues at 4-aligned position g (relative to `res`) and translate
// them: byte j -> symbol, or 0xFF when g+j is outside [b, e).
__device__ __forceinline__ uint32_t load_symbols(const uint8_t *__restrict__ res, int64_t nres,
                                                 int64_t g, int64_t b, int64_t e,
                                                 const uint8_t *s_lut) {
    if (g >= e || g + 4 <= b) return 0xFFFFFFFFu;
    uint32_t w;
    if (g + 4 <= nres) {
        w = __ldg(reinterpret_cast<const uint32_t *>(res + g));
    } else {
        w = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (g + j < nres) w |= uint32_t(res[g + j]) << (8 * j);
    }
    uint32_t out = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t byte = (w >> (8 * j)) & 0xFFu;
        uint32_t s = s_lut[byte];
        const int64_t p = g + j;
        if (p < b || p >= e) s = SYM_INVALID;
        out |= s << (8 * j);
    }
    return out;
}

// One warp enumerates every window start of sequence [b, e).
//   emit(gpos, code, ok) is called by every lane for its 4 positions per step
//   (also for invalid ones, ok = false), in converged code, so emit may use
//   warp collectives.  gpos is the position of the window start in `res`.
template <typename CodeT, int NW, typename Emit>
__device__ __forceinline__ void warp_scan_sequence(const uint8_t *__restrict__ res, int64_t nres,
                                                   int64_t b, int64_t e, const uint8_t *s_lut,
                                                   int nsym, int k, Emit &&emit) {
    const int lane = threadIdx.x & 31;
    if (e - b < k) return;
    const int64_t last = e - k;               // last valid window start
    const int64_t c0 = b & ~int64_t(3);
    uint32_t prev = load_symbols(res, nres, c0 + 4 * lane, b, e, s_lut);
    for (int64_t c = c0; c <= last; c += 128) {
        const uint32_t cur = load_symbols(res, nres, c + 128 + 4 * lane, b, e, s_lut);
        uint32_t w[NW + 1];
        w[0] = prev;
#pragma unroll
        for (int j = 1; j <= NW; ++j) {
            const uint32_t src = (lane >= j) ? prev : cur;
            w[j] = __shfl_sync(FULL, src, (lane + j) & 31);
        }
        CodeT code[4] = {0, 0, 0, 0};
        bool bad[4] = {false, false, false, false};
#pragma unroll
        for (int j = 0; j < 4 * NW + 4; ++j) {
            const uint32_t s = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
            const bool inv = (s == SYM_INVALID);
            const CodeT v = inv ? CodeT(0) : CodeT(s);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (j >= t && j < t + k) {      // warp-uniform predicate
                    code[t] = code[t] * CodeT(nsym) + v;
                    bad[t] |= inv;
                }
            }
        }
        const int64_t g = c + 4 * lane;
#pragma unroll
        for (int t = 0; t < 4; ++t) emit(g + t, code[t], !bad[t]);
        prev = cur;
    }
}

// Dispatch helper: NW is a template parameter, k a run-time value.
#define SKM_DISPATCH_NW(nw, ...)                                  \
    switch (nw) {                                                 \
        case 1: { constexpr int NW = 1; __VA_ARGS__; } break;     \
        case 2: { constexpr int NW = 2; __VA_ARGS__; } break;     \
        case 4: { constexpr int NW = 4; __VA_ARGS__; } break;     \
        case 8: { constexpr int NW = 8; __VA_ARGS__; } break;     \
        default: { constexpr int NW = 16; __VA_ARGS__; } break;   \
    }

// nsym^k as unsigned 128-bit-safe computation: returns false on overflow of 2^64.
inline bool code_space(int nsym, int k, unsigned __int128 *out) {
    unsigned __int128 s = 1;
    for (int i = 0; i < k; ++i) {
        s *= (unsigned)nsym;
        if (s > ((unsigned __int128)1 << 64)) return false;
    }
    *out = s;
    return true;
}

// host: workspace regions start on 256-byte boundaries
inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }
// host: smallest b in [1, 64] with 2^b >= n (the radix-sort bits that hold every value below n)
inline int bits_for(unsigned __int128 n) { int b = 1; while (b < 64 && (((unsigned __int128)1) << b) < n) ++b; return b; }

// column of `code` in a basis given as its ascending code list and the column of every entry; -1 when absent
__device__ __forceinline__ int32_t lookup_column(const uint64_t *__restrict__ sorted_codes, const int32_t *__restrict__ col_of_sorted,
                                                 int64_t K, uint64_t code) {
    int64_t lo = 0, hi = K;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(sorted_codes + mid) < code) lo = mid + 1; else hi = mid;
    }
    return (lo < K && __ldg(sorted_codes + lo) == code) ? __ldg(col_of_sorted + lo) : -1;
}

// basis lookup: sorted code list + column of each entry; `bucket` (nullable) = start index of every 2^shift-wide
// code range, so the binary search runs over a handful of entries
struct SortedBasis {
    const uint64_t *codes;
    const int32_t *col;
    const uint32_t *bucket;     // [nbucket + 1]
    int64_t K;
    int shift;
};
__device__ __forceinline__ int32_t sorted_lookup(const SortedBasis &b, uint64_t code) {
    int64_t lo = 0, hi = b.K;
    if (b.bucket) {
        const uint64_t q = code >> b.shift;
        lo = __ldg(b.bucket + q);
        hi = __ldg(b.bucket + q + 1);
    }
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(b.codes + mid) < code) lo = mid + 1; else hi = mid;
    }
    return (lo < b.K && __ldg(b.codes + lo) == code) ? __ldg(b.col + lo) : -1;
}

constexpr int SORTED_BUCKET_BITS = 20;
// bytes of the bucket index sorted_basis_init may build
constexpr size_t SORTED_BUCKET_BYTES = ((size_t(1) << SORTED_BUCKET_BITS) + 2) * 4;
// host (skm_csrsort.cu): *sb = the lookup over (codes, col, K) in a code space of S codes; bases of more than 64 entries
// get a bucket index of at most 2^20 + 1 entries, built into `bucket` (SORTED_BUCKET_BYTES) on stream st
int sorted_basis_init(SortedBasis *sb, const uint64_t *codes, const int32_t *col, int64_t K, unsigned __int128 S,
                      uint32_t *bucket, cudaStream_t st);

int check_common(const void *d_residues, int64_t nres, const void *d_offsets, int64_t nseq,
                 const void *d_lut, int nsym, int k);

}  // namespace skm
