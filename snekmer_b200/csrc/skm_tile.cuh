// skm_tile.cuh — CTA-level segment scanner: the inner loop of kernels (a), (b), (b').
//
// A CTA walks a CONTIGUOUS range of the packed residue buffer in segments of at
// most `seg_cap` residues.  Per segment:
//   1. stage   residues are read once from HBM with aligned 16-byte loads,
//              translated through the 256-byte alphabet LUT and written to
//              shared memory as one symbol byte per residue
//                 bits 0-5  digit (index of the reduced symbol, 0 if invalid)
//                 bit  6    SYM_BAD   residue has no symbol (X, B, Z, *, lower case ...)
//                 bit  7    SYM_FLAG  first residue of a sequence
//   2. flag    the sequence starts that fall in the segment are marked;
//   3. scan    every thread owns a contiguous chunk of C positions (C = 4*odd,
//              so the 32 lanes of a warp hit 32 different banks) and rolls the
//              base-|A| code of the window ENDING at each position:
//                 code = code*|A| + digit[i]            -> emit if run >= k
//                 code -= digit[i-k+1] * |A|^(k-1)
//              `run` counts the valid residues since the last invalid residue
//              or sequence start, so windows never cross a sequence boundary
//              or an unmapped residue (vectorize.py:239-249).  A chunk warms up
//              on the k-1 symbols in front of it; the k-1 symbols in front of a
//              segment are carried over from the previous one in shared memory.
// The rare path (invalid residue / sequence start, ~0.4 % of positions) is a
// divergent branch; the common path is a dozen instructions per residue.
#pragma once

#include "skm_common.cuh"

namespace skm {

constexpr int TS_THREADS = 256;                    // upper bound of the CTA size of scanner kernels
constexpr int TS_PAD = 64;                         // >= k-1 halo symbols in front of the segment
constexpr int TS_MAX_K = TS_PAD;                   // k-1 <= 63
constexpr int TS_MAX_NSYM = 64;                    // digits are 6 bits
constexpr uint32_t SYM_BAD = 0x40u, SYM_FLAG = 0x80u, SYM_DIGIT = 0x3Fu;

// shared bytes of a symbol buffer that stages up to seg_cap residues (seg_cap % 16 == 0)
__host__ __device__ constexpr int ts_sym_bytes(int seg_cap) { return TS_PAD + seg_cap + 32; }
// segment capacity when every one of `threads` threads owns at most c residues (c = 4 * odd)
__host__ __device__ constexpr int ts_seg_cap(int c, int threads = TS_THREADS) { return threads * c; }

// chunk length for n positions over the CTA's threads: smallest 4*odd >= ceil(n / threads)
__device__ __forceinline__ int ts_chunk(int n) {
    int c = (n + int(blockDim.x) - 1) / int(blockDim.x);
    c = (c + 3) >> 2;            // words
    c |= 1;                      // odd
    return c << 2;
}

// ---- shared-memory accessors on 32-bit shared-window addresses --------------------
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
template <int OFF>
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF));
    return v;
}
__device__ __forceinline__ void reds_add_u32(uint32_t a, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void reds_min_u32(uint32_t a, uint32_t v) {
    asm volatile("red.shared.min.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// LUT with the in-kernel symbol encoding (digit | SYM_BAD)
__device__ __forceinline__ void ts_lut_init(uint8_t *s_lut, const uint8_t *__restrict__ lut) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        const uint32_t v = lut[i];
        s_lut[i] = (v == SYM_INVALID) ? uint8_t(SYM_BAD) : uint8_t(v);
    }
}

__device__ __forceinline__ uint32_t ts_translate4(uint32_t w, const uint8_t *s_lut) {
    return uint32_t(s_lut[w & 0xFFu]) | (uint32_t(s_lut[(w >> 8) & 0xFFu]) << 8) |
           (uint32_t(s_lut[(w >> 16) & 0xFFu]) << 16) | (uint32_t(s_lut[w >> 24]) << 24);
}

// Geometry of one staged segment [a, b) (absolute positions in `res`).
struct TsSeg {
    int64_t base;   // absolute position of symbol index TS_PAD (16-byte aligned)
    int lo, hi;     // symbol indices of a and b
};

// Step 1 of a segment: translate [a & ~15, b) into s_sym[TS_PAD ...).  For every segment
// but the first of a range, `a` is 16-byte aligned and the caller has already moved the
// previous tail into the pad (ts_tail_read / ts_tail_write).
__device__ __forceinline__ TsSeg ts_stage(const uint8_t *__restrict__ res, int64_t nres, int64_t a, int64_t b,
                                          const uint8_t *s_lut, uint8_t *s_sym) {
    TsSeg g;
    g.base = a & ~int64_t(15);
    g.lo = TS_PAD + int(a - g.base);
    g.hi = g.lo + int(b - a);
    const int nvec = int((b - g.base + 15) >> 4);
    uint4 *dst = reinterpret_cast<uint4 *>(s_sym + TS_PAD);
    for (int v = threadIdx.x; v < nvec; v += blockDim.x) {
        const int64_t p = g.base + 16 * int64_t(v);
        uint4 x;
        if (p + 16 <= nres) {
            x = __ldg(reinterpret_cast<const uint4 *>(res + p));
        } else {
            uint32_t w[4] = {0, 0, 0, 0};
            for (int j = 0; j < 16; ++j)
                if (p + j < nres) w[j >> 2] |= uint32_t(res[p + j]) << (8 * (j & 3));
            x = make_uint4(w[0], w[1], w[2], w[3]);
        }
        x.x = ts_translate4(x.x, s_lut);
        x.y = ts_translate4(x.y, s_lut);
        x.z = ts_translate4(x.z, s_lut);
        x.w = ts_translate4(x.w, s_lut);
        dst[v] = x;
    }
    return g;
}

// After the staging stores are visible (one __syncthreads): for the first segment of a
// range, everything in front of `a` reads as invalid.
__device__ __forceinline__ void ts_invalidate_front(uint8_t *s_sym, const TsSeg &g) {
    for (int i = threadIdx.x; i < g.lo; i += blockDim.x) s_sym[i] = uint8_t(SYM_BAD);
}

// Between two segments: read the last k-1 symbols of the finished segment ...
__device__ __forceinline__ uint32_t ts_tail_read(const uint8_t *s_sym, const TsSeg &g, int k) {
    const int t = threadIdx.x;
    return (t < k - 1) ? s_sym[g.hi - (k - 1) + t] : 0u;
}
// ... and, after a __syncthreads, put them in front of the next one.
__device__ __forceinline__ void ts_tail_write(uint8_t *s_sym, uint32_t v, int k) {
    const int t = threadIdx.x;
    if (t < k - 1) s_sym[TS_PAD - (k - 1) + t] = uint8_t(v);
}

// One position of the scan.  p = shared address of symbol i, q = p - (k-1).
//   emit(p, code, ok)  window ENDING at p; ok = it is valid (starts at p-(k-1));
//                      called for every position so that it can stay branch-free
//   boundary(p)        symbol at p is the first residue of a sequence (before emit)
template <int OFF, typename CodeT, typename Emit, typename Boundary>
__device__ __forceinline__ void ts_step(uint32_t p, uint32_t q, uint32_t k, CodeT nsym, CodeT neg_pow_k1, uint32_t &run,
                                        CodeT &code, Emit &emit, Boundary &boundary) {
    uint32_t s = lds_u8<OFF>(p);
    if (s >= SYM_BAD) {
        if (s & SYM_FLAG) { run = 0u; boundary(p + OFF); }
        if (s & SYM_BAD) run = 0xFFFFFFFFu;
        s &= SYM_DIGIT;
    }
    run += 1;
    code = code * nsym + CodeT(s);
    emit(p + OFF, code, run >= k);
    code += CodeT(lds_u8<OFF>(q) & SYM_DIGIT) * neg_pow_k1;
}

// Step 3 for one thread: symbol indices [i0, i1) of the staged segment at shared address `sym`.
template <typename CodeT, typename Emit, typename Boundary>
__device__ __forceinline__ void ts_scan_chunk(uint32_t sym, int i0, int i1, int k, CodeT nsym, CodeT pow_k1, Emit &&emit,
                                              Boundary &&boundary) {
    if (i0 >= i1) return;
    uint32_t run = 0;
    CodeT code = 0;
    uint32_t p = sym + uint32_t(i0 - (k - 1));
    for (int j = 0; j < k - 1; ++j, ++p) {
        uint32_t s = lds_u8<0>(p);
        if (s >= SYM_BAD) {
            run = (s & SYM_BAD) ? 0xFFFFFFFFu : 0u;
            s &= SYM_DIGIT;
        }
        run += 1;
        code = code * nsym + CodeT(s);
    }
    const CodeT npow = CodeT(0) - pow_k1;
    const uint32_t uk = uint32_t(k);
    uint32_t q = p - (uk - 1u);
    const uint32_t pend = sym + uint32_t(i1);
    for (; p + 4 <= pend; p += 4, q += 4) {
        ts_step<0>(p, q, uk, nsym, npow, run, code, emit, boundary);
        ts_step<1>(p, q, uk, nsym, npow, run, code, emit, boundary);
        ts_step<2>(p, q, uk, nsym, npow, run, code, emit, boundary);
        ts_step<3>(p, q, uk, nsym, npow, run, code, emit, boundary);
    }
    for (; p < pend; ++p, ++q) ts_step<0>(p, q, uk, nsym, npow, run, code, emit, boundary);
}

__device__ __forceinline__ int64_t lower_bound_off(const int64_t *__restrict__ off, int64_t n, int64_t target) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(off + mid) < target) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Part i of `parts` owns the sequences whose start lies in [R*i/parts, R*(i+1)/parts) of the residue span R:
// contiguous and residue-balanced.  Part 0 starts at sequence 0 and the last part ends at nseq.
__device__ __forceinline__ void seq_range(const int64_t *__restrict__ off, int64_t nseq, int64_t part, int64_t parts,
                                          int64_t *lo, int64_t *hi) {
    const int64_t r0 = __ldg(off), span = __ldg(off + nseq) - r0;
    const auto start = [&](int64_t i) { return lower_bound_off(off, nseq, r0 + (int64_t)(((__int128)span * i) / parts)); };
    *lo = (part == 0) ? 0 : start(part);
    *hi = (part + 1 == parts) ? nseq : start(part + 1);
}

template <int GT> __device__ __forceinline__ void gsync() { if (GT == 32) __syncwarp(); else __syncthreads(); }

constexpr int TS_WALK_C = 12;                      // residues per thread and segment of ts_group_walk (4 * odd)

// ---- a group of GT threads (one warp, or a whole CTA) walks ONE sequence [b, e) byte-wise -------------------------
// Segments of GT * TS_WALK_C residues are staged into s_sym (ts_sym_bytes of that, at shared address sym_addr) through
// the LUT, one 16-byte vector per thread; the first segment's front reads as invalid, the k-1 symbols in front of every
// later segment are carried over from the previous one.  Thread g owns a 4*odd chunk of every segment, warms up on the
// k-1 symbols in front of it and rolls the code with a run counter.  emit(widx, code, ok) is called at every position
// of the chunk: widx = index of the window ending there (window i covers residues b+i .. b+i+k-1; negative in front of
// the first window), ok = the window is valid (never for widx < 0).  All GT threads call this, converged.
template <int GT, int UNROLL, typename KeyT, typename Emit>
__device__ __forceinline__ void ts_group_walk(const uint8_t *__restrict__ res, int64_t nres, int64_t b, int64_t e,
                                              const uint8_t *s_lut, uint8_t *s_sym, uint32_t sym_addr, int k, KeyT nsym,
                                              KeyT pow_k1, int g, Emit &&emit) {
    constexpr int SEG = GT * TS_WALK_C;
    const uint32_t uk = uint32_t(k);
    bool first = true;
    uint32_t tail0 = 0, tail1 = 0;                      // the last k-1 symbols of the previous segment (k-1 <= 63)
    for (int64_t a = b; a < e;) {
        const int64_t a2 = min(e, (a + SEG) & ~int64_t(15));
        if (!first) {
            if (g < k - 1) s_sym[TS_PAD - (k - 1) + g] = uint8_t(tail0);
            if (g + 32 < k - 1) s_sym[TS_PAD - (k - 1) + g + 32] = uint8_t(tail1);
        }
        // stage: [a & ~15, a2) translated into s_sym[TS_PAD ...), one 16-byte vector per thread
        const int64_t base = a & ~int64_t(15);
        const int lo_i = TS_PAD + int(a - base), hi_i = lo_i + int(a2 - a);
        const int nvec = int((a2 - base + 15) >> 4);
        if (g < nvec) {
            const int64_t p = base + 16 * int64_t(g);
            uint4 x;
            if (p + 16 <= nres) {
                x = __ldg(reinterpret_cast<const uint4 *>(res + p));
            } else {
                uint32_t w4[4] = {0, 0, 0, 0};
                for (int j = 0; j < 16; ++j)
                    if (p + j < nres) w4[j >> 2] |= uint32_t(res[p + j]) << (8 * (j & 3));
                x = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            }
            x.x = ts_translate4(x.x, s_lut);
            x.y = ts_translate4(x.y, s_lut);
            x.z = ts_translate4(x.z, s_lut);
            x.w = ts_translate4(x.w, s_lut);
            reinterpret_cast<uint4 *>(s_sym + TS_PAD)[g] = x;
        }
        gsync<GT>();
        if (first) {                                    // nothing in front of the sequence start is a residue of it
            for (int i = g; i < lo_i; i += GT) s_sym[i] = uint8_t(SYM_BAD);
            gsync<GT>();
        }
        // scan: thread g owns symbols [i0, i1), warms up on the k-1 symbols in front of them
        const int n = hi_i - lo_i;
        const int C = ((int(unsigned(n + GT - 1) / GT) + 3) >> 2 | 1) << 2;     // smallest 4 * odd >= ceil(n / GT)
        const int i0 = lo_i + g * C, i1 = min(i0 + C, hi_i);
        if (i0 < i1) {
            uint32_t run = 0;
            KeyT code = 0;
            uint32_t p = sym_addr + uint32_t(i0) - (uk - 1u);
            for (uint32_t j = 1; j < uk; ++j, ++p) {
                const uint32_t sy = lds_u8<0>(p);
                run = (sy >= SYM_BAD) ? 0u : run + 1u;
                code = code * nsym + KeyT(sy);
            }
            const uint32_t pend = sym_addr + uint32_t(i1);
            const uint32_t back = uk - 1u;
            int64_t widx = (a - b) + int64_t(i0 - lo_i) - int64_t(k - 1);
#pragma unroll UNROLL
            for (; p < pend; ++p, ++widx) {
                const uint32_t sy = lds_u8<0>(p);
                run = (sy >= SYM_BAD) ? 0u : run + 1u;
                code = code * nsym + KeyT(sy);
                emit(widx, code, run >= uk);
                code -= KeyT(lds_u8<0>(p - back)) * pow_k1;
            }
        }
        gsync<GT>();
        if (g < k - 1) tail0 = s_sym[hi_i - (k - 1) + g];
        if (g + 32 < k - 1) tail1 = s_sym[hi_i - (k - 1) + g + 32];
        gsync<GT>();
        first = false;
        a = a2;
    }
}

// ---- a CTA walks its share of the residue buffer, with the sequence index of every window -----------
// Used by the kernels that need to know WHICH sequence a window belongs to while scanning a long
// contiguous range (key generation for the sort-based sparse paths).  CTA i owns the sequences that
// start in the i-th 1/gridDim of the buffer.  emit(rel_end, row, code, ok) is called for EVERY residue
// position of the range: rel_end = position of the window's last residue minus `origin`,
// row = index of the sequence that holds it, ok = the window is valid.
// emit also receives the index of the position inside the staged segment (0 .. n-1), and post(rel_a, n) is called by
// ALL threads after every segment's scan (behind a barrier; another barrier follows): kernels that write one value per
// position stage the values in shared memory in emit and copy them out coalesced in post — a thread's own positions
// are 52 apart from its neighbour's, so direct global stores are fully uncoalesced.
// s_sym: ts_sym_bytes(seg_cap) bytes; s_lut: 256 bytes (ts_lut_init done, barrier passed);
// s_ctl: 4 x int64 of shared scratch.
template <typename CodeT, typename Emit, typename Post>
__device__ __forceinline__ void ts_range_scan_rows(const uint8_t *__restrict__ res, int64_t nres,
                                                   const int64_t *__restrict__ off, int64_t nseq, const uint8_t *s_lut,
                                                   uint8_t *s_sym, int seg_cap, int k, CodeT nsym, CodeT pow_k1,
                                                   int64_t origin, int64_t *s_ctl, Emit &&emit, Post &&post) {
    const int tid = threadIdx.x;
    unsigned int *s_nstart = reinterpret_cast<unsigned int *>(s_ctl + 2);
    if (tid == 0) { seq_range(off, nseq, blockIdx.x, gridDim.x, &s_ctl[0], &s_ctl[1]); *s_nstart = 0; }
    __syncthreads();
    const int64_t lo = s_ctl[0], hi = s_ctl[1];
    if (lo >= hi) return;
    uint32_t sym_addr = smem_addr(s_sym);
    asm volatile("" : "+r"(sym_addr));
    const int64_t r_lo = __ldg(off + lo), r_hi = __ldg(off + hi);
    int64_t cur = lo;                 // first sequence that starts at or after `a`
    bool first = true;
    uint32_t tail = 0;
    for (int64_t a = r_lo; a < r_hi;) {
        const int64_t b = min(r_hi, (a + seg_cap) & ~int64_t(15));
        if (!first) ts_tail_write(s_sym, tail, k);
        const TsSeg g = ts_stage(res, nres, a, b, s_lut, s_sym);
        __syncthreads();
        if (first) ts_invalidate_front(s_sym, g);
        unsigned int mine = 0;
        for (int64_t s = cur + tid; s < hi; s += blockDim.x) {
            const int64_t o = __ldg(off + s);
            if (o >= b) break;
            s_sym[g.lo + int(o - a)] |= uint8_t(SYM_FLAG);
            ++mine;
        }
        if (mine) atomicAdd(s_nstart, mine);
        __syncthreads();
        const int64_t nstart = *s_nstart;
        const int C = ts_chunk(g.hi - g.lo);
        const int i0 = g.lo + tid * C, i1 = min(i0 + C, g.hi);
        if (i0 < i1) {
            // sequence holding position x0 = a + (i0 - g.lo): the last one of [cur-1, cur+nstart) that starts at or before x0
            const int64_t x0 = a + (i0 - g.lo);
            int64_t l = cur, h = cur + nstart;               // count of sequences in [cur, cur+nstart) with off <= x0 ...
            while (l < h) {
                const int64_t mid = (l + h) >> 1;
                if (__ldg(off + mid) < x0) l = mid + 1; else h = mid;   // ... strictly before x0: a start AT x0 is flagged
            }
            int64_t row = l - 1;
            const int64_t to_abs = (g.base - TS_PAD) - int64_t(sym_addr);    // absolute position = shared address + to_abs
            const int64_t to_rel = to_abs - origin;
            const uint32_t seg0 = sym_addr + uint32_t(g.lo);           // shared address of the segment's first symbol
            ts_scan_chunk<CodeT>(
                sym_addr, i0, i1, k, nsym, pow_k1,
                [&](uint32_t p, CodeT code, bool ok) { emit(int64_t(p) + to_rel, row, code, ok, int(p - seg0)); },
                [&](uint32_t p) {
                    const int64_t pos = int64_t(p) + to_abs;
                    do { ++row; } while (row + 1 < nseq && __ldg(off + row + 1) <= pos);   // skips empty sequences
                });
        }
        tail = ts_tail_read(s_sym, g, k);
        __syncthreads();
        post(a - origin, g.hi - g.lo);
        first = false;
        cur += nstart;
        a = b;
        __syncthreads();
        if (tid == 0) *s_nstart = 0;    // ordered before the next atomicAdd by the barrier after staging
    }
}

inline bool ts_supported(int nsym, int k) { return nsym <= TS_MAX_NSYM && k <= TS_MAX_K; }

// ---- bulk (TMA engine) shared -> global store -------------------------------------
// All threads that wrote the source call ts_bulk_fence() and then __syncthreads(); ONE
// thread calls ts_bulk_store() (dst, src 16-byte aligned, bytes % 16 == 0) and
// ts_bulk_wait_read() before the source is overwritten.
__device__ __forceinline__ void ts_bulk_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void ts_bulk_store(void *gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void ts_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

}  // namespace skm
