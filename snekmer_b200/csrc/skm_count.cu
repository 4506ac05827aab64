// skm_count.cu — kernel (b): per-sequence k-mer counts over the basis.
//
// Dense path (skm_count_dense) — replaces the per-sequence loops of
// kmerize.smk:117-120 (np.isin presence), learn.smk:359-383 and
// apply.smk:195-206 (dict counts gathered in basis order):
//   a CTA owns a tile of T consecutive sequences and keeps all T count rows in
//   shared memory as packed 16-bit (or 32-bit) counters; its warps pull
//   sequences off a shared-memory ticket, walk them with warp_scan_sequence and
//   bump row[col_of_code[code]] with shared-memory atomics; the tile is then
//   streamed to HBM as ONE contiguous range (rows are adjacent in the [N,K]
//   output) with 16-byte stores while the counters are re-zeroed in place.
//   HBM traffic is the algorithmic minimum: every residue read once, every
//   output element written once.  Algorithmic bytes per sequence:
//   L + 8 + K*sizeof(out).
//
// Sparse paths (skm_count_csr, 32-bit keys = columns; skm_count_csr_wide, 64-bit codes with an optional sorted
// basis): window keys -> segmented radix sort of each sequence's keys -> run-length encode into CSR.  Both are the
// cross-checks of skm_count_csr_sorted (skm_csrsort.cu).
#include <cstring>
#include <type_traits>

#include <cub/cub.cuh>

#include "skm_common.cuh"
#include "skm_tile.cuh"

namespace skm {

// ---------------------------------------------------------------------------
// dense
// ---------------------------------------------------------------------------
constexpr int CD_MAX_ROWS = 32;   // rows (sequences) per tile

// counters live in shared memory in the OUTPUT layout (int32, or uint16 packed two per word), so a tile
// is flushed with one bulk shared->global copy
template <typename OutT> struct cnt_ops;
template <> struct cnt_ops<int32_t> {
    static __device__ __forceinline__ void add(uint32_t base, uint32_t idx) { reds_add_u32(base + (idx << 2), 1u); }
};
template <> struct cnt_ops<uint16_t> {
    // no carry into the upper half while a count stays < 65536 (host: max_len <= 65535)
    static __device__ __forceinline__ void add(uint32_t base, uint32_t idx) {
        reds_add_u32(base + ((idx >> 1) << 2), 1u << ((idx & 1u) << 4));
    }
};

// smem: [T*K counters of OutT | symbol buffer for seg_cap residues]
template <typename OutT, bool HAS_MAP>
__global__ void __launch_bounds__(TS_THREADS) count_dense_kernel(const uint8_t *__restrict__ res, int64_t nres,
                                                                 const int64_t *__restrict__ off, int64_t nseq,
                                                                 const uint8_t *__restrict__ lut, uint32_t nsym, int k,
                                                                 uint32_t pow_k1, const int32_t *__restrict__ col_of_code,
                                                                 int K, int T, int seg_cap, OutT *__restrict__ out) {
    extern __shared__ __align__(128) uint8_t s_raw[];
    __shared__ uint8_t s_lut[256];
    __shared__ int32_t s_off[CD_MAX_ROWS + 1];        // row starts relative to the tile
    const int64_t tile_elems = int64_t(T) * K;
    const uint32_t cnt_bytes = uint32_t((size_t(tile_elems) * sizeof(OutT) + 15) & ~size_t(15));
    uint4 *s_cnt4 = reinterpret_cast<uint4 *>(s_raw);
    uint8_t *s_sym = s_raw + cnt_bytes;
    uint32_t cnt_addr = smem_addr(s_raw), sym_addr = smem_addr(s_sym);
    asm volatile("" : "+r"(cnt_addr), "+r"(sym_addr));      // keep the window addresses in registers
    ts_lut_init(s_lut, lut);
    for (int i = threadIdx.x; i < int(cnt_bytes >> 4); i += blockDim.x) s_cnt4[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const int tid = threadIdx.x;
    const int64_t ntiles = (nseq + T - 1) / T;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t s0 = tile * T;
        const int rows = (nseq - s0 < T) ? int(nseq - s0) : T;
        const int64_t r0 = __ldg(off + s0), r1 = __ldg(off + s0 + rows);
        for (int r = tid; r <= rows; r += blockDim.x) s_off[r] = int32_t(__ldg(off + s0 + r) - r0);
        bool first = true;
        uint32_t tail = 0;
        for (int64_t a = r0; a < r1;) {
            const int64_t b = min(r1, (a + seg_cap) & ~int64_t(15));
            if (!first) ts_tail_write(s_sym, tail, k);
            const TsSeg g = ts_stage(res, nres, a, b, s_lut, s_sym);
            __syncthreads();
            if (first) ts_invalidate_front(s_sym, g);
            const int a_rel = int(a - r0), b_rel = int(b - r0);
            for (int r = tid; r < rows; r += blockDim.x) {
                const int o = s_off[r];
                if (o >= a_rel && o < b_rel) s_sym[g.lo + (o - a_rel)] |= uint8_t(SYM_FLAG);
            }
            __syncthreads();
            const int C = ts_chunk(g.hi - g.lo);
            const int i0 = g.lo + tid * C, i1 = min(i0 + C, g.hi);
            if (i0 < i1) {
                const int shift = a_rel - g.lo;                 // tile-relative position = symbol index + shift
                const int rel0 = i0 + shift;
                int lo = 0, hi = rows;                          // rows that start strictly before rel0
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (s_off[mid] < rel0) lo = mid + 1; else hi = mid;
                }
                int row = lo - 1;                               // -1 only when i0 is the (flagged) tile start
                uint32_t row_base = uint32_t(row) * uint32_t(K);
                const int shift_addr = shift - int(sym_addr);   // tile-relative position = shared address + shift_addr
                ts_scan_chunk<uint32_t>(
                    sym_addr, i0, i1, k, nsym, pow_k1,
                    [&](uint32_t, uint32_t code, bool ok) {
                        int32_t col = -1;
                        if (ok) col = HAS_MAP ? __ldg(col_of_code + code) : int32_t(code);
                        if (col >= 0) cnt_ops<OutT>::add(cnt_addr, row_base + uint32_t(col));
                    },
                    [&](uint32_t p) {
                        const int rel = int(p) + shift_addr;
                        do { ++row; } while (s_off[row + 1] <= rel);   // skips empty sequences; s_off[rows] > rel
                        row_base = uint32_t(row) * uint32_t(K);
                    });
            }
            tail = ts_tail_read(s_sym, g, k);
            first = false;
            a = b;
            __syncthreads();
        }
        // ---- flush: the tile is one contiguous range of the [N, K] output ----
        ts_bulk_fence();
        __syncthreads();
        OutT *dst = out + s0 * K;
        const int64_t n_elems = int64_t(rows) * K;
        const OutT *s_cnt = reinterpret_cast<const OutT *>(s_raw);
        if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
            const uint32_t bytes = uint32_t(n_elems * sizeof(OutT)) & ~15u;
            if (tid == 0 && bytes) ts_bulk_store(dst, cnt_addr, bytes);
            for (int64_t i = bytes / sizeof(OutT) + tid; i < n_elems; i += blockDim.x) dst[i] = s_cnt[i];
            if (tid == 0) ts_bulk_wait_read();
        } else {
            for (int64_t i = tid; i < n_elems; i += blockDim.x) dst[i] = s_cnt[i];
        }
        __syncthreads();
        for (int i = tid; i < int(cnt_bytes >> 4); i += blockDim.x) s_cnt4[i] = make_uint4(0u, 0u, 0u, 0u);
        // the next tile touches the counters only after two more barriers
    }
}

// ---------------------------------------------------------------------------
// dense, one warp per sequence (rows up to ~9 KB)
// ---------------------------------------------------------------------------
// The tile kernel above synchronises the whole CTA four times per tile (stage / flag / scan / flush): at K = 1000
// it spends 28 % of its time in barriers and reaches 61 % of HBM.  Here every WARP is its own pipeline: it owns a
// contiguous, residue-balanced range of sequences, a private counter row (the output layout) and a private symbol
// buffer in shared memory, and only ever executes __syncwarp.  A sequence is walked in segments of 384 residues
// (12 per lane; the mean protein fits one segment); the finished row leaves with one bulk shared->global copy.
// ~48 independent warps per SM hide each other's load, bulk-store and shared-atomic latencies.
constexpr int CW_WARPS = 8;
constexpr int CW_SEG = 32 * TS_WALK_C;
constexpr int CW_SYM = ts_sym_bytes(CW_SEG);      // 480

// MAP: 0 = identity basis (column = code), 1 = col_of_code staged in shared memory as uint16 columns (S <= 16384;
// filtered codes point at a dummy counter behind the row, so the scan needs no validity test), 2 = col_of_code read
// from global memory (large code spaces), 3 = MAP 1's columns in lane-striped words (small S, count_dense_warp_kernel
// only): word w of lane l sits at byte (w * 32 + l) * 4 and holds entries 2w and 2w + 1, so every lane reads its own
// bank and a warp's map read is one shared-memory wavefront instead of ~4.3 at random codes.
// The scan is written out here rather than through ts_scan_chunk: one sequence per warp needs no boundary handling,
// symbols are used raw (an invalid symbol's garbage digit is added and later subtracted with the same value, and no
// window containing it is ever emitted), and the column comes from shared memory: 13 SASS instructions per residue
// against 24 for the generic scanner.
template <typename OutT, int MAP>
__device__ __forceinline__ void cw_emit(uint32_t code, uint32_t cnt_addr, uint32_t col_addr, const int32_t *__restrict__ col_of_code, int K) {
    uint32_t col;
    if (MAP == 0) col = code;
    else if (MAP == 1) asm volatile("ld.shared.u16 %0, [%1];" : "=r"(col) : "r"(col_addr + 2u * code));
    else { const int32_t c = __ldg(col_of_code + code); col = c >= 0 ? uint32_t(c) : uint32_t(K); }
    cnt_ops<OutT>::add(cnt_addr, col);
}

// Branch-free emission: an invalid window is counted into the dummy counter behind the row (MAP 0: column K; MAP 1
// and 3: the extra map entry S points at it), so the compiler can issue LDS + ATOMS without a branch around them.
// MAP 3: col_addr is the map's shared address plus 4 * lane.
template <typename OutT, int MAP>
__device__ __forceinline__ void cw_emit_sel(uint32_t code, bool ok, uint32_t cnt_addr, uint32_t col_addr,
                                            const int32_t *__restrict__ col_of_code, int S, int K) {
    if (MAP == 2) {
        if (ok) cw_emit<OutT, 2>(code, cnt_addr, col_addr, col_of_code, K);
        return;
    }
    uint32_t col;
    if (MAP == 0) {
        col = ok ? code : uint32_t(K);
    } else if (MAP == 1) {
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(col) : "r"(col_addr + 2u * (ok ? code : uint32_t(S))));
    } else {
        const uint32_t c = ok ? code : uint32_t(S);      // entry c: byte (c >> 1) * 128 + (c & 1) * 2 = c * 2 + (c >> 1) * 124
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(col) : "r"(col_addr + 2u * c + 124u * (c >> 1)));
    }
    cnt_ops<OutT>::add(cnt_addr, col);
}

// Zero `bytes` (a multiple of 8) of shared memory from shared address `addr` with one st.bulk (SASS UMEMSETS) instead
// of 16-byte stores from every lane.  st.bulk has no completion mechanism of its own: it is a weak store of the generic
// proxy, ordered against the other lanes' later shared-memory atomics by the __syncwarp / __syncthreads that follows.
__device__ __forceinline__ void cw_zero_row(uint32_t addr, uint32_t bytes) {
    asm volatile("st.bulk.weak.shared::cta [%0], %1, 0;" ::"r"(addr), "l"(uint64_t(bytes)) : "memory");
}

// Column of basis entry i for the shared map: K (the dummy counter) for codes outside the basis and for entry S,
// where invalid windows go.
__device__ __forceinline__ uint32_t cw_map_entry(const int32_t *__restrict__ col_of_code, int i, int S, int K) {
    const int32_t c = i < S ? __ldg(col_of_code + i) : -1;
    return uint32_t(c >= 0 ? c : K);
}

// Column map (MAP 1 or 3) and this warp's zeroed counter row, before the kernel's one CTA-wide barrier.
template <int MAP>
__device__ __forceinline__ void cw_prologue(uint8_t *s_map, const int32_t *__restrict__ col_of_code, int S, int K,
                                            uint32_t cnt_addr, uint32_t row_bytes, int lane) {
    if (MAP == 1) {
        uint16_t *s_col = reinterpret_cast<uint16_t *>(s_map);
        for (int i = threadIdx.x; i <= S; i += blockDim.x) s_col[i] = uint16_t(cw_map_entry(col_of_code, i, S, K));
    } else if (MAP == 3) {
        uint32_t *s_words = reinterpret_cast<uint32_t *>(s_map);
        const int nwords = (S + 2) >> 1;                                        // entries 0 .. S
        for (int i = threadIdx.x; i < nwords * 32; i += blockDim.x) {
            const int e = (i >> 5) * 2;
            s_words[i] = cw_map_entry(col_of_code, e, S, K) | (cw_map_entry(col_of_code, e + 1, S, K) << 16);
        }
    }
    if (lane == 0) cw_zero_row(cnt_addr, row_bytes);
}

// Flush the finished row to dst (one contiguous K * sizeof(OutT) range of the output) and re-zero it.  Lane 0 zeroes
// the row after the bulk copy has read it (cp.async.bulk.wait_group.read in the same thread).
template <typename OutT>
__device__ __forceinline__ void cw_flush_row(OutT *dst, const uint8_t *mine, uint32_t cnt_addr, int K, uint32_t row_bytes,
                                             int bulk_ok, int lane) {
    if (bulk_ok) {
        ts_bulk_fence();
        __syncwarp();
        if (lane == 0) { ts_bulk_store(dst, cnt_addr, uint32_t(K) * uint32_t(sizeof(OutT))); ts_bulk_wait_read(); }
    } else {
        __syncwarp();
        const OutT *s_cnt = reinterpret_cast<const OutT *>(mine);
        for (int i = lane; i < K; i += 32) dst[i] = s_cnt[i];
        __syncwarp();
    }
    if (lane == 0) cw_zero_row(cnt_addr, row_bytes);
    __syncwarp();
}

// PRMT in its sign mode: byte i of the result is 0xFF where bit 7 of byte i of x is set, else 0.
__device__ __forceinline__ uint32_t cw_sign_bytes(uint32_t x) {
    uint32_t r;
    asm("prmt.b32 %0, %1, 0, 0xBA98;" : "=r"(r) : "r"(x));
    return r;
}

// PRMT with a selector whose nibbles are known to be < 8 (__byte_perm masks them with 0x7777 first)
__device__ __forceinline__ uint32_t cw_prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// Four residue bytes -> four symbols (digit or SYM_BAD), for a LUT that maps every byte outside 0x40-0x5F to SYM_BAD
// (upper-case letters and @[\]^_; every built-in alphabet but ptm).  L holds the LUT entries 0x40-0x5F, four per
// register.  One PRMT per register pair picks by the low 3 bits of each byte, two byte-mask muxes by bits 3 and 4,
// and bytes whose top three bits are not 010 become SYM_BAD: ~20 ALU instructions against four LDS.U8.
__device__ __forceinline__ uint32_t cw_translate_reg(uint32_t raw, const uint32_t (&L)[8]) {
    const uint32_t s = raw & 0x07070707u;
    const uint32_t sel = __byte_perm(s | (s >> 4), 0u, 0x0020u);                // nibble i = low 3 bits of byte i
    const uint32_t q0 = cw_prmt(L[0], L[1], sel), q1 = cw_prmt(L[2], L[3], sel);
    const uint32_t q2 = cw_prmt(L[4], L[5], sel), q3 = cw_prmt(L[6], L[7], sel);
    const uint32_t m3 = cw_sign_bytes(raw << 4), m4 = cw_sign_bytes(raw << 3);   // bytes with bit 3 / bit 4 set
    const uint32_t lo = (q0 & ~m3) | (q1 & m3), hi = (q2 & ~m3) | (q3 & m3);
    const uint32_t t = (lo & ~m4) | (hi & m4);
    const uint32_t y = raw ^ 0x40404040u;
    const uint32_t bad = cw_sign_bytes(y | (y << 1) | (y << 2));                // any of bits 5-7 of byte ^ 0x40 set
    return (t & ~bad) | (SYM_BAD * 0x01010101u & bad);
}

// First version of the warp kernel (round 1): translated symbols staged as bytes, two LDS.U8 per residue, a run
// counter (ts_group_walk).  The path for k - 1 > 4.
template <typename OutT, int MAP>
__global__ void __launch_bounds__(32 * CW_WARPS, 6)
count_dense_warp_bytes_kernel(const uint8_t *__restrict__ res, int64_t nres, const int64_t *__restrict__ off, int64_t nseq,
                              const uint8_t *__restrict__ lut, uint32_t nsym, int k, uint32_t pow_k1,
                              const int32_t *__restrict__ col_of_code, int S, int K, uint32_t row_bytes, uint32_t map_bytes, int bulk_ok,
                              OutT *__restrict__ out) {
    extern __shared__ __align__(128) uint8_t s_raw[];
    __shared__ uint8_t s_lut[256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *mine = s_raw + map_bytes + size_t(warp) * (row_bytes + CW_SYM);
    uint8_t *s_sym = mine + row_bytes;
    uint32_t cnt_addr = smem_addr(mine), sym_addr = smem_addr(s_sym), col_addr = smem_addr(s_raw);   // map: [S + 1] uint16 when MAP == 1
    asm volatile("" : "+r"(cnt_addr), "+r"(sym_addr), "+r"(col_addr));      // keep the window addresses in registers
    ts_lut_init(s_lut, lut);
    cw_prologue<MAP>(s_raw, col_of_code, S, K, cnt_addr, row_bytes, lane);
    __syncthreads();                                        // LUT and column map; the only CTA-wide barrier
    // this warp's sequences: those that start in the w-th 1/W of the residue buffer
    int64_t lo = 0, hi = 0;
    if (lane == 0) seq_range(off, nseq, int64_t(blockIdx.x) * CW_WARPS + warp, int64_t(gridDim.x) * CW_WARPS, &lo, &hi);
    lo = __shfl_sync(FULL, lo, 0);
    hi = __shfl_sync(FULL, hi, 0);
    int64_t e = (lo < hi) ? __ldg(off + lo) : 0;
    for (int64_t s = lo; s < hi; ++s) {
        const int64_t b = e;
        e = __ldg(off + s + 1);
        ts_group_walk<32, 4, uint32_t>(res, nres, b, e, s_lut, s_sym, sym_addr, k, nsym, pow_k1, lane, [&](int64_t, uint32_t code, bool ok) {
            if (ok) cw_emit<OutT, MAP>(code, cnt_addr, col_addr, col_of_code, K);
        });
        cw_flush_row(out + s * K, mine, cnt_addr, K, row_bytes, bulk_ok, lane);
    }
}

// Round-2 warp kernel (k - 1 <= 4, i.e. every dense basis of practical size).  What changed against the first version
// (profiles/r1m_* -> R2b_* -> R2c_*): 700 warp instructions and 221 shared-memory wavefronts per sequence, 59 % of the
// instructions OUTSIDE the scan loop (staging the translated symbols: 96; 64-bit position arithmetic per sequence and
// segment: ~170).
//   * the RAW residue bytes are staged (one LDG.128 + STS.128 per lane) and translated inside the scan, one LDS.U8 from
//     the LUT per residue, straight into the register that feeds the rolling code: no translate-and-repack pass;
//   * a lane owns a 4-ALIGNED chunk and reads it as 32-bit words; the translated previous word stays in a register and
//     one funnel shift of (previous : current) gives the four symbols that leave the window: no second read per residue;
//   * no run counter and no branch: the 8 validity bits of (previous : current) are tested against a k-bit window mask
//     and the emission is predicated (a branch on "any invalid byte" diverges in 54 % of the warp iterations — first
//     word, last word, an X somewhere in 192 bytes — and made the first word-based version execute MORE instructions);
//   * positions are 32-bit offsets from the warp's own (16-byte aligned) base, and the offsets of 31 sequences are
//     fetched with one coalesced load and handed out by shuffles;
// Round 3 (profiles/count_dense_*, DESIGN 3.2) took the LSU wavefronts that are not the counter atomics off the
// shared-memory pipe: the flushed row is re-zeroed with one st.bulk from lane 0 (cw_zero_row) instead of 8 STS.128 per
// lane; for a LUT whose entries outside 0x40-0x5F are all SYM_BAD the residues are translated in registers
// (cw_translate_reg) instead of four LDS.U8 per word; for small S the column map is lane-striped (MAP 3), which needs
// one CTA of up to 32 warps per SM for its 4 * 32 bytes per map word.
// Measured and dropped (profiles/R2e_*): re-zeroing the flushed row with the copy engine (cp.async.bulk shared -> shared
// from a zero row needs a cluster launch and ran at 1.21 ms against 0.85 ms; global (L2) -> shared 0.92 ms).
template <typename OutT, int MAP>
__global__ void __launch_bounds__(MAP == 3 ? 1024 : 32 * CW_WARPS, MAP == 3 ? 1 : 6)
count_dense_warp_kernel(const uint8_t *__restrict__ res, int64_t nres, const int64_t *__restrict__ off, int64_t nseq,
                        const uint8_t *__restrict__ lut, uint32_t nsym, int k, uint32_t pow_k1,
                        const int32_t *__restrict__ col_of_code, int S, int K, uint32_t row_bytes, uint32_t map_bytes, int bulk_ok,
                        OutT *__restrict__ out) {
    extern __shared__ __align__(128) uint8_t s_raw[];
    __shared__ __align__(16) uint8_t s_lut[256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    uint8_t *mine = s_raw + map_bytes + size_t(warp) * (row_bytes + CW_SYM);
    uint8_t *s_res = mine + row_bytes;                                           // raw residue bytes of the segment
    uint32_t cnt_addr = smem_addr(mine), raw_addr = smem_addr(s_res), lut_addr = smem_addr(s_lut);
    uint32_t col_addr = smem_addr(s_raw) + (MAP == 3 ? 4u * uint32_t(lane) : 0u);
    asm volatile("" : "+r"(cnt_addr), "+r"(raw_addr), "+r"(col_addr), "+r"(lut_addr));
    ts_lut_init(s_lut, lut);                                                     // invalid bytes -> SYM_BAD (0x40)
    if (threadIdx.x == 0) s_lut[0] = uint8_t(SYM_BAD);                           // byte 0 pads the staged segment: never a symbol
    bool lut_in_regs = true;                                                     // every entry outside 0x40-0x5F is SYM_BAD
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if ((i & 0xE0) != 0x40 && i != 0 && lut[i] != SYM_INVALID) lut_in_regs = false;
    cw_prologue<MAP>(s_raw, col_of_code, S, K, cnt_addr, row_bytes, lane);
    const bool reg_lut = __syncthreads_and(lut_in_regs);    // LUT and column map; the only CTA-wide barrier
    // this warp's sequences: those that start in the w-th 1/W of the residue buffer
    int64_t lo = 0, hi = 0;
    if (lane == 0) seq_range(off, nseq, int64_t(blockIdx.x) * nwarps + warp, int64_t(gridDim.x) * nwarps, &lo, &hi);
    lo = __shfl_sync(FULL, lo, 0);
    hi = __shfl_sync(FULL, hi, 0);
    if (lo >= hi) return;
    // 32-bit positions relative to the 16-byte aligned base of this warp's range (alignment of a position is preserved)
    const int64_t r_base = __ldg(off + lo) & ~int64_t(15);
    const uint8_t *__restrict__ resw = res + r_base;
    const int64_t lim64 = nres - r_base;                    // bytes that may be read from resw
    const uint32_t lim = lim64 > int64_t(0xFFFFFFF0u) ? 0xFFFFFFF0u : uint32_t(lim64);
    const uint32_t uk = uint32_t(k), km1 = uk - 1u;
    const uint32_t out_shift = 32u - 8u * km1;              // (previous : current) >> out_shift = the four outgoing symbols
    const uint32_t win0 = ((1u << uk) - 1u) << (4u - km1);  // validity bits a window ending at byte 0 of `current` covers
    const uint32_t npow = 0u - pow_k1;
    uint32_t L[8];                                          // LUT entries 0x40-0x5F (used when reg_lut)
    {
        const uint4 a = reinterpret_cast<const uint4 *>(s_lut + 0x40)[0], b = reinterpret_cast<const uint4 *>(s_lut + 0x40)[1];
        L[0] = a.x; L[1] = a.y; L[2] = a.z; L[3] = a.w; L[4] = b.x; L[5] = b.y; L[6] = b.z; L[7] = b.w;
    }
    // the whole walk, once per translation (a uniform branch: every warp of the CTA takes the same one)
    auto walk = [&](auto use_regs) {
        constexpr bool REG = decltype(use_regs)::value;
        // the four symbols of a word, packed and one by one
        auto translate = [&](uint32_t raw, uint32_t (&t)[4]) -> uint32_t {
            if (REG) {
                const uint32_t T = cw_translate_reg(raw, L);
                t[0] = T & 0xFFu; t[1] = __byte_perm(T, 0u, 0x4441u); t[2] = __byte_perm(T, 0u, 0x4442u); t[3] = T >> 24;
                return T;
            }
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t[0]) : "r"(lut_addr + __byte_perm(raw, 0u, 0x4440u)));
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t[1]) : "r"(lut_addr + __byte_perm(raw, 0u, 0x4441u)));
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t[2]) : "r"(lut_addr + __byte_perm(raw, 0u, 0x4442u)));
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t[3]) : "r"(lut_addr + __byte_perm(raw, 0u, 0x4443u)));
            return t[0] | (t[1] << 8) | (t[2] << 16) | (t[3] << 24);
        };
        uint32_t tailw = 0;
        for (int64_t s0 = lo; s0 < hi; s0 += 31) {
            // one coalesced load of 32 offsets: sequences s0 .. s0+30 (b = rel[i], e = rel[i+1])
            const int64_t si = min(s0 + lane, hi);
            const uint32_t rel = uint32_t(__ldg(off + si) - r_base);
            const int ns = (hi - s0 < 31) ? int(hi - s0) : 31;
            for (int i = 0; i < ns; ++i) {
                const uint32_t b = __shfl_sync(FULL, rel, i), e = __shfl_sync(FULL, rel, i + 1);
                bool first = true;
                for (uint32_t a = b; a < e;) {
                    const uint32_t a2 = min(e, (a + uint32_t(CW_SEG)) & ~15u);
                    const uint32_t base = a & ~15u;
                    const int lo_i = TS_PAD + int(a - base), hi_i = lo_i + int(a2 - a);
                    const int nvec = int((a2 - base + 15u) >> 4);
                    // stage the raw bytes [base, a2) at s_res[TS_PAD ...): one 16-byte vector per lane (at most 25)
                    if (lane < nvec) {
                        const uint32_t p = base + 16u * uint32_t(lane);
                        uint4 x;
                        if (p + 16u <= lim) {
                            x = __ldg(reinterpret_cast<const uint4 *>(resw + p));
                        } else {
                            uint32_t w4[4] = {0, 0, 0, 0};
                            for (int j = 0; j < 16; ++j)
                                if (p + uint32_t(j) < lim) w4[j >> 2] |= uint32_t(resw[p + j]) << (8 * (j & 3));
                            x = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                        }
                        reinterpret_cast<uint4 *>(s_res + TS_PAD)[lane] = x;
                    }
                    if (!first && lane == 0) reinterpret_cast<uint32_t *>(s_res)[TS_PAD / 4 - 1] = tailw;   // the 4 bytes in front of this segment
                    __syncwarp();
                    // byte 0 translates to SYM_BAD: everything in front of the sequence and behind the segment's last word is invalid
                    if (first) { const int f0 = (lo_i & ~3) - 4; if (f0 + lane < lo_i) s_res[f0 + lane] = 0; }   // previous word + front of the first word
                    if (lane < ((4 - (hi_i & 3)) & 3)) s_res[hi_i + lane] = 0;
                    __syncwarp();
                    // lane owns cw words (cw odd -> conflict-free LDS.32) from word index w0
                    const int A = lo_i & ~3;
                    const int n = hi_i - A;
                    const int cw = (((n + 31) >> 5) + 3) >> 2 | 1;
                    const int w0 = (A >> 2) + lane * cw, w1 = min(w0 + cw, (hi_i + 3) >> 2);
                    if (w0 < w1) {
                        uint32_t pa = raw_addr + 4u * uint32_t(w0);
                        uint32_t raw;
                        asm volatile("ld.shared.u32 %0, [%1+-4];" : "=r"(raw) : "r"(pa));
                        uint32_t t[4];
                        uint32_t prevT = translate(raw, t);
                        uint32_t pinv = (((prevT >> 6) & 0x01010101u) * 0x01020408u) >> 24;      // bit i: byte i of prevT is no symbol
                        uint32_t code = 0;
                        for (uint32_t t = 0; t < km1; ++t) code = code * nsym + ((prevT >> (out_shift + 8u * t)) & 0xFFu);
                        for (int w = w0; w < w1; ++w, pa += 4u) {
                            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(raw) : "r"(pa));
                            const uint32_t curT = translate(raw, t);
                            const uint32_t outw = __funnelshift_rc(prevT, curT, out_shift);
                            const uint32_t cinv = (((curT >> 6) & 0x01010101u) * 0x01020408u) >> 24;
                            const uint32_t inv8 = pinv | (cinv << 4);
                            code = code * nsym + t[0];
                            cw_emit_sel<OutT, MAP>(code, (inv8 & win0) == 0u, cnt_addr, col_addr, col_of_code, S, K);
                            code = __byte_perm(outw, 0u, 0x4440u) * npow + code;
                            code = code * nsym + t[1];
                            cw_emit_sel<OutT, MAP>(code, (inv8 & (win0 << 1)) == 0u, cnt_addr, col_addr, col_of_code, S, K);
                            code = __byte_perm(outw, 0u, 0x4441u) * npow + code;
                            code = code * nsym + t[2];
                            cw_emit_sel<OutT, MAP>(code, (inv8 & (win0 << 2)) == 0u, cnt_addr, col_addr, col_of_code, S, K);
                            code = __byte_perm(outw, 0u, 0x4442u) * npow + code;
                            code = code * nsym + t[3];
                            cw_emit_sel<OutT, MAP>(code, (inv8 & (win0 << 3)) == 0u, cnt_addr, col_addr, col_of_code, S, K);
                            code = __byte_perm(outw, 0u, 0x4443u) * npow + code;
                            prevT = curT;
                            pinv = cinv;
                        }
                    }
                    __syncwarp();
                    if (a2 < e && lane == 0) tailw = reinterpret_cast<const uint32_t *>(s_res)[(hi_i >> 2) - 1];   // hi_i is 16-aligned here
                    __syncwarp();
                    first = false;
                    a = a2;
                }
                cw_flush_row(out + (s0 + i) * K, mine, cnt_addr, K, row_bytes, bulk_ok, lane);
            }
        }
    };
    // the register translation needs the 1024-thread CTA's 64 registers: at 40 the walk spills
    if (MAP == 3 && reg_lut) walk(std::true_type{});
    else walk(std::false_type{});
}

// Everything a dense count launch passes to its kernel besides the launch shape.
struct DenseArgs {
    const uint8_t *res;
    int64_t nres;
    const int64_t *off;
    int64_t nseq;
    const uint8_t *lut;
    uint32_t nsym;
    int k;
    uint32_t pow_k1;
    const int32_t *col_of_code;
    int S, K;
    void *out;
    cudaStream_t st;
};

constexpr int CD_THREADS = 128;   // threads of the tile kernel

template <typename OutT>
static int launch_dense_tile(const DenseArgs &a, int grid, size_t smem, int T, int seg_cap) {
    const auto kern = a.col_of_code ? count_dense_kernel<OutT, true> : count_dense_kernel<OutT, false>;
    SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, CD_THREADS, smem, a.st>>>(a.res, a.nres, a.off, a.nseq, a.lut, a.nsym, a.k, a.pow_k1, a.col_of_code, a.K, T,
                                           seg_cap, static_cast<OutT *>(a.out));
    SKM_LAUNCH_CHECK("count_dense_kernel");
    return SKM_OK;
}

// words: the round-2 kernel (k - 1 <= 4), else the byte-wise one; map_mode selects MAP (3: words only)
template <typename OutT>
static int launch_dense_warp(const DenseArgs &a, bool words, int map_mode, int grid, int warps, size_t smem, uint32_t row_bytes,
                             uint32_t map_bytes, int bulk_ok) {
    using Kern = decltype(&count_dense_warp_kernel<OutT, 0>);
    const Kern kerns[2][4] = {{count_dense_warp_bytes_kernel<OutT, 0>, count_dense_warp_bytes_kernel<OutT, 1>, count_dense_warp_bytes_kernel<OutT, 2>, nullptr},
                              {count_dense_warp_kernel<OutT, 0>, count_dense_warp_kernel<OutT, 1>, count_dense_warp_kernel<OutT, 2>, count_dense_warp_kernel<OutT, 3>}};
    const Kern kern = kerns[words][map_mode];
    SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 32 * warps, smem, a.st>>>(a.res, a.nres, a.off, a.nseq, a.lut, a.nsym, a.k, a.pow_k1, a.col_of_code, a.S,
                                           a.K, row_bytes, map_bytes, bulk_ok, static_cast<OutT *>(a.out));
    SKM_LAUNCH_CHECK(words ? "count_dense_warp_kernel" : "count_dense_warp_bytes_kernel");
    return SKM_OK;
}

// ---------------------------------------------------------------------------
// sparse (CSR): the two segmented-sort paths, 32-bit and 64-bit keys
// ---------------------------------------------------------------------------
// One warp per sequence over its sorted keys: count the runs (fill = false: rowptr[s + 1] = runs of row s) or write them
// at rowptr[s] (fill = true).  32-bit keys (already columns) always go to keys_out.  64-bit keys: with a sorted basis,
// runs whose code it does not hold are dropped and the column of every run goes to cols_out; keys_out and cols_out
// may each be NULL.
template <typename KeyT>
__global__ void __launch_bounds__(256) csr_runs_kernel(const KeyT *__restrict__ keys, const int64_t *__restrict__ off,
                                                       int64_t nseq, const uint64_t *__restrict__ sorted_codes,
                                                       const int32_t *__restrict__ col_of_sorted, int64_t K, bool fill,
                                                       int64_t *__restrict__ rowptr, KeyT *__restrict__ keys_out,
                                                       uint32_t *__restrict__ cols_out, int32_t *__restrict__ vals) {
    constexpr KeyT NONE = code_traits<KeyT>::none;
    constexpr bool WIDE = sizeof(KeyT) == 8;       // 32-bit keys: no basis, the keys are the output
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    for (int64_t s = warp; s < nseq; s += nwarps) {
        const int64_t b = __ldg(off + s), e = __ldg(off + s + 1);
        int64_t nrun = 0;
        const int64_t wbase = fill ? rowptr[s] : 0;
        for (int64_t p0 = b; p0 < e; p0 += 32) {
            const int64_t p = p0 + lane;
            const KeyT key = (p < e) ? keys[p] : NONE;
            const KeyT prevk = (p > b && p < e) ? keys[p - 1] : NONE;
            bool head = (p < e) && key != NONE && (p == b || key != prevk);
            int32_t col = -1;
            if (WIDE && head && sorted_codes) { col = lookup_column(sorted_codes, col_of_sorted, K, key); head = col >= 0; }
            const unsigned m = __ballot_sync(FULL, head);
            if (fill && head) {
                int64_t q = p + 1;
                while (q < e && keys[q] == key) ++q;       // runs are short: a k-mer repeated within one protein
                const int64_t slot = wbase + nrun + __popc(m & ((1u << lane) - 1u));
                if (!WIDE || keys_out) keys_out[slot] = key;
                if (WIDE && cols_out) cols_out[slot] = uint32_t(col);
                vals[slot] = int32_t(q - p);
            }
            nrun += __popc(m);
        }
        if (!fill && lane == 0) rowptr[s + 1] = nrun;
    }
}

// skm_wide.cu: argument checks of the 64-bit paths and the 64-bit key of every window
int wide_check(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
               int nsym, int k, const char *who, unsigned __int128 *S);
int launch_window_codes64(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
                          int nsym, int k, uint64_t *d_keys, cudaStream_t st);

}  // namespace skm

extern "C" int skm_window_keys_u32(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                                   const uint8_t *d_lut, int nsym, int k, const int32_t *d_col_of_code, uint32_t *d_keys,
                                   cudaStream_t st);   // skm_sparse.cu

extern "C" {

int skm_count_dense(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                    const uint8_t *d_lut, int nsym, int k, const int32_t *d_col_of_code, int64_t S, int64_t K,
                    int out_bits, void *d_counts, int64_t max_len, skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (S128 > (unsigned __int128)SKM_DENSE_MAX_SPACE || (int64_t)S128 != S) {
        set_error("skm_count_dense: S=%lld must equal nsym^k and be <= 2^27", (long long)S);
        return S128 > (unsigned __int128)SKM_DENSE_MAX_SPACE ? SKM_ERR_UNSUPPORTED : SKM_ERR_INVALID;
    }
    if (out_bits != 32 && out_bits != 16) { set_error("skm_count_dense: out_bits must be 32 or 16"); return SKM_ERR_INVALID; }
    if (!d_col_of_code && K != S) { set_error("skm_count_dense: identity basis needs K == S"); return SKM_ERR_INVALID; }
    if (K < 0 || K > S) { set_error("skm_count_dense: K=%lld out of range", (long long)K); return SKM_ERR_INVALID; }
    if (out_bits == 16 && (max_len <= 0 || max_len > 65535)) { set_error("skm_count_dense: uint16 output needs 0 < max_len <= 65535"); return SKM_ERR_INVALID; }
    if (nseq == 0 || K == 0) return SKM_OK;
    if (!d_counts) { set_error("skm_count_dense: d_counts is NULL"); return SKM_ERR_INVALID; }
    if (!ts_supported(nsym, k)) { set_error("skm_count_dense: nsym=%d k=%d outside the kernel envelope (nsym <= %d, k <= %d)", nsym, k, TS_MAX_NSYM, TS_MAX_K); return SKM_ERR_UNSUPPORTED; }
    if ((reinterpret_cast<uintptr_t>(d_counts) & 15u) != 0) { set_error("skm_count_dense: d_counts must be 16-byte aligned"); return SKM_ERR_INVALID; }
    const size_t out_bytes = out_bits / 8;
    const size_t smem_cap = 200 * 1024;
    if (size_t(K) * out_bytes > smem_cap) {
        set_error("skm_count_dense: K=%lld rows do not fit shared memory; use skm_count_csr", (long long)K);
        return SKM_ERR_UNSUPPORTED;
    }
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    const DenseArgs args{d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k, pow_k1, d_col_of_code, (int)S, (int)K,
                         d_counts, (cudaStream_t)stream};
    // Rows up to ~9 KB: one warp per sequence with a private counter row (>= 24 warps per SM).  One extra (dummy)
    // counter behind the row absorbs the windows whose code is filtered out of the basis.
    const uint32_t row_bytes = uint32_t((size_t(K + 1) * out_bytes + 15) & ~size_t(15));
    if (row_bytes + CW_SYM <= 9 * 1024 + 256 && K < 65535) {
        int map_mode = !d_col_of_code ? 0 : (S <= 16384 ? 1 : 2);
        const bool words = k - 1 <= 4;
        const int bulk_ok = ((size_t(K) * out_bytes) % 16 == 0) ? 1 : 0;
        const size_t per_warp = row_bytes + CW_SYM;
        // MAP 3 (lane-striped map): one CTA per SM with as many warps as fit next to the map, if that is at least 24
        // (the uint16 map with 5-6 CTAs of 8 warps keeps ~40 warps per SM to hide latency; the striped shape was
        // measured at 32).  C2 (S = K = 1000, int32): 64 KB of map + 32 warps, 208 KB.
        const size_t cta_smem = 227 * 1024 - 256;                                   // minus the static LUT
        const uint32_t striped_bytes = uint32_t(size_t((S + 2) / 2) * 128);
        if (map_mode == 1 && words && striped_bytes + 24 * per_warp <= cta_smem) {
            map_mode = 3;
            const int warps = (int)std::min<size_t>(32, (cta_smem - striped_bytes) / per_warp);
            const size_t smem = striped_bytes + size_t(warps) * per_warp;
            const int grid = (int)std::min<int64_t>((nseq + warps - 1) / warps, int64_t(sm_count()));
            return out_bits == 32 ? launch_dense_warp<int32_t>(args, true, 3, grid, warps, smem, row_bytes, striped_bytes, bulk_ok)
                                  : launch_dense_warp<uint16_t>(args, true, 3, grid, warps, smem, row_bytes, striped_bytes, bulk_ok);
        }
        const uint32_t map_bytes = map_mode == 1 ? uint32_t((size_t(S + 1) * 2 + 127) & ~size_t(127)) : 0u;     // + the entry for invalid windows
        const size_t smem_w = map_bytes + size_t(CW_WARPS) * per_warp;
        int per_sm_w = int((227 * 1024) / (smem_w + 1024 + 256));
        if (per_sm_w > 6) per_sm_w = 6;
        if (per_sm_w < 1) per_sm_w = 1;
        const int grid_w = (int)std::min<int64_t>((nseq + CW_WARPS - 1) / CW_WARPS, int64_t(sm_count()) * per_sm_w);
        return out_bits == 32 ? launch_dense_warp<int32_t>(args, words, map_mode, grid_w, CW_WARPS, smem_w, row_bytes, map_bytes, bulk_ok)
                              : launch_dense_warp<uint16_t>(args, words, map_mode, grid_w, CW_WARPS, smem_w, row_bytes, map_bytes, bulk_ok);
    }
    // Tile shape.  Many small CTAs per SM (each with its own tile in flight) hide the staging-load, barrier
    // and bulk-store latencies of one another: 128 threads, ~16 KB of counters, rows a multiple of
    // 4 (int32) / 8 (uint16) so that every tile start is 16-byte aligned and leaves as one bulk copy.
    int64_t align_rows = 16 / (int64_t)out_bytes;           // rows per 16 bytes of output in the worst case ...
    while (align_rows > 1 && (size_t(align_rows / 2) * K * out_bytes) % 16 == 0) align_rows /= 2;   // ... fewer when K allows
    int64_t T = int64_t((16 * 1024) / (size_t(K) * out_bytes));
    if (T >= align_rows) T -= T % align_rows;
    if (T < align_rows) T = (size_t(align_rows) * K * out_bytes <= 64 * 1024) ? align_rows : 1;
    if (T > CD_MAX_ROWS) T = CD_MAX_ROWS;
    const int seg_cap = ts_seg_cap(28, CD_THREADS);
    const size_t sym_bytes = (size_t)ts_sym_bytes(seg_cap);
    const size_t sm_bytes = 227 * 1024, per_cta_reserved = 1024 + 512;
    const size_t smem = ((size_t(T) * K * out_bytes + 15) & ~size_t(15)) + sym_bytes;
    const int64_t ntiles = (nseq + T - 1) / T;
    int per_sm = int(sm_bytes / (smem + per_cta_reserved));
    if (per_sm > 2048 / CD_THREADS) per_sm = 2048 / CD_THREADS;
    if (per_sm > 32) per_sm = 32;
    if (per_sm < 1) per_sm = 1;
    const int grid = (int)std::min<int64_t>(ntiles, int64_t(sm_count()) * per_sm);
    return out_bits == 32 ? launch_dense_tile<int32_t>(args, grid, smem, (int)T, seg_cap)
                          : launch_dense_tile<uint16_t>(args, grid, smem, (int)T, seg_cap);
}

// cub::DeviceSegmentedSort takes 32-bit item counts: one call handles < 2^30 residues (callers shard above that).
static const int64_t CSR_MAX_RES = (1ll << 30);

// workspace of one segmented sort of key_bytes-wide keys: two key buffers and the larger of the sort's and the scan's temp
static size_t csr_segsort_workspace(int64_t nres, int64_t nseq, size_t key_bytes) {
    using namespace skm;
    if (nres <= 0 || nseq <= 0) return 256;
    const int items = (int)std::min<int64_t>(nres, CSR_MAX_RES), segs = (int)std::min<int64_t>(nseq, (1ll << 31) - 1);
    size_t t_sort = 0, t_scan = 0;
    if (key_bytes == 8)
        cub::DeviceSegmentedSort::SortKeys(nullptr, t_sort, (const uint64_t *)nullptr, (uint64_t *)nullptr, items, segs,
                                           (const int64_t *)nullptr, (const int64_t *)nullptr);
    else
        cub::DeviceSegmentedSort::SortKeys(nullptr, t_sort, (const uint32_t *)nullptr, (uint32_t *)nullptr, items, segs,
                                           (const int64_t *)nullptr, (const int64_t *)nullptr);
    cub::DeviceScan::InclusiveSum(nullptr, t_scan, (const int64_t *)nullptr, (int64_t *)nullptr, nseq);
    return 2 * align256((size_t)nres * key_bytes) + align256(std::max(t_sort, t_scan)) + 1024;
}

size_t skm_count_csr_workspace(int64_t nres, int64_t nseq) { return csr_segsort_workspace(nres, nseq, 4); }

int skm_count_csr(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                  const uint8_t *d_lut, int nsym, int k, const int32_t *d_col_of_code, int64_t S,
                  int64_t *d_rowptr, uint32_t *d_cols, int32_t *d_vals, void *workspace, size_t workspace_bytes,
                  skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (S128 >= ((unsigned __int128)1 << 32)) { set_error("skm_count_csr: code space must be < 2^32 (32-bit keys)"); return SKM_ERR_UNSUPPORTED; }
    if (d_col_of_code && (int64_t)S128 != S) { set_error("skm_count_csr: S must equal nsym^k"); return SKM_ERR_INVALID; }
    if (!d_rowptr) { set_error("skm_count_csr: d_rowptr is NULL"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_rowptr, 0, 8 * (size_t)(nseq + 1), st));
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!d_cols || !d_vals) { set_error("skm_count_csr: d_cols / d_vals are NULL"); return SKM_ERR_INVALID; }
    if (nres >= CSR_MAX_RES || nseq >= (1ll << 31)) { set_error("skm_count_csr: more than 2^30 residues per call; split the shard"); return SKM_ERR_UNSUPPORTED; }
    const size_t need = skm_count_csr_workspace(nres, nseq);
    if (!workspace || workspace_bytes < need) { set_error("skm_count_csr: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    const size_t seg = align256((size_t)nres * 4);
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    uint32_t *keys_a = (uint32_t *)p, *keys_b = (uint32_t *)(p + seg);
    void *temp = p + 2 * seg;
    size_t temp_bytes = workspace_bytes - (size_t)((char *)temp - (char *)workspace);
    if (!ts_supported(nsym, k)) { set_error("skm_count_csr: nsym=%d k=%d outside the kernel envelope", nsym, k); return SKM_ERR_UNSUPPORTED; }
    const int grid = sm_count() * 8;
    // keys are indexed by the absolute position of the window's last residue (positions outside every sequence
    // are never read by the segmented sort)
    rc = skm_window_keys_u32(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, d_col_of_code, keys_a, st);
    if (rc) return rc;
    SKM_CUDA_TRY(cub::DeviceSegmentedSort::SortKeys(temp, temp_bytes, keys_a, keys_b, (int)nres, (int)nseq, d_offsets,
                                                    d_offsets + 1, st));
    csr_runs_kernel<uint32_t><<<grid, 256, 0, st>>>(keys_b, d_offsets, nseq, nullptr, nullptr, 0, false, d_rowptr, nullptr, nullptr, nullptr);
    SKM_LAUNCH_CHECK("csr_runs_kernel(count)");
    temp_bytes = workspace_bytes - (size_t)((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceScan::InclusiveSum(temp, temp_bytes, d_rowptr + 1, d_rowptr + 1, nseq, st));
    csr_runs_kernel<uint32_t><<<grid, 256, 0, st>>>(keys_b, d_offsets, nseq, nullptr, nullptr, 0, true, d_rowptr, d_cols, nullptr, d_vals);
    SKM_LAUNCH_CHECK("csr_runs_kernel(fill)");
    return SKM_OK;
}

size_t skm_count_csr_wide_workspace(int64_t nres, int64_t nseq) { return csr_segsort_workspace(nres, nseq, 8); }

int skm_count_csr_wide(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                       const uint8_t *d_lut, int nsym, int k, const uint64_t *d_sorted_codes,
                       const int32_t *d_col_of_sorted, int64_t K, int64_t *d_rowptr, uint64_t *d_codes_out,
                       uint32_t *d_cols_out, int32_t *d_vals, void *workspace, size_t workspace_bytes,
                       skm_stream_t stream) {
    using namespace skm;
    unsigned __int128 S;
    int rc = wide_check(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, "skm_count_csr_wide", &S);
    if (rc) return rc;
    if (!d_rowptr) { set_error("skm_count_csr_wide: d_rowptr is NULL"); return SKM_ERR_INVALID; }
    if (d_sorted_codes && (!d_col_of_sorted || K < 0)) { set_error("skm_count_csr_wide: basis given without its column map"); return SKM_ERR_INVALID; }
    if (d_cols_out && !d_sorted_codes) { set_error("skm_count_csr_wide: d_cols_out needs a basis"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_rowptr, 0, 8 * (size_t)(nseq + 1), st));
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!d_vals || (!d_codes_out && !d_cols_out)) { set_error("skm_count_csr_wide: NULL output"); return SKM_ERR_INVALID; }
    const size_t need = skm_count_csr_wide_workspace(nres, nseq);
    if (!workspace || workspace_bytes < need) { set_error("skm_count_csr_wide: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(nres) * 8);
    uint64_t *keys_a = (uint64_t *)p, *keys_b = (uint64_t *)(p + seg);
    void *temp = p + 2 * seg;
    const size_t temp_cap = workspace_bytes - (size_t)((char *)temp - (char *)workspace);
    size_t temp_bytes = temp_cap;
    // keys are indexed by the absolute position of the window's last residue; positions outside every sequence are
    // never read by the segmented sort
    rc = launch_window_codes64(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, keys_a, st);
    if (rc) return rc;
    SKM_CUDA_TRY(cub::DeviceSegmentedSort::SortKeys(temp, temp_bytes, keys_a, keys_b, (int)nres, (int)nseq, d_offsets, d_offsets + 1, st));
    const int grid = sm_count() * 8;
    csr_runs_kernel<uint64_t><<<grid, 256, 0, st>>>(keys_b, d_offsets, nseq, d_sorted_codes, d_col_of_sorted, K, false, d_rowptr, nullptr, nullptr, nullptr);
    SKM_LAUNCH_CHECK("csr_runs_kernel(count)");
    temp_bytes = temp_cap;
    SKM_CUDA_TRY(cub::DeviceScan::InclusiveSum(temp, temp_bytes, d_rowptr + 1, d_rowptr + 1, nseq, st));
    csr_runs_kernel<uint64_t><<<grid, 256, 0, st>>>(keys_b, d_offsets, nseq, d_sorted_codes, d_col_of_sorted, K, true, d_rowptr, d_codes_out, d_cols_out, d_vals);
    SKM_LAUNCH_CHECK("csr_runs_kernel(fill)");
    return SKM_OK;
}

}  // extern "C"
