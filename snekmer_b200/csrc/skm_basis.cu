// skm_basis.cu — kernel (b'): k-mer basis construction (kmerize.smk:89-104).
//
// Pass 1 of the reference's vectorize rule builds {kmer: total count} in
// first-occurrence (dict insertion) order and keeps count > min_filter.  Here:
//   skm_basis_accumulate  count[c] += 1, first[c] = min(global position) over
//                         all valid windows, for the code space S = nsym^k;
//   skm_basis_finalize    keep count > min_filter, order by `first`.
// Keeping `first` as the global residue position (res_base + index in the
// packed buffer) makes shards mergeable by (sum, min) — the multi-GPU exchange.
//
// Small code spaces (S <= SMALL_S) are privatised per CTA in shared memory
// (counts and first positions relative to the CTA's contiguous residue range)
// and flushed with S atomics per CTA; large ones go straight to L2 atomics
// (low contention because the table is large) with a read-before-min filter.
// Algorithmic bytes: R residues + 8 (N+1) offsets + 24 S table.
#include <algorithm>

#include <cub/cub.cuh>

#include "skm_common.cuh"
#include "skm_tile.cuh"

namespace skm {

constexpr int64_t SMALL_S = 16384;   // 8 B per code of shared memory -> 128 KB

constexpr int BS_SEG = ts_seg_cap(52);              // residues per staged segment (52 per thread)
constexpr int BS_SYM_BYTES = ts_sym_bytes(BS_SEG);

// One kernel for both table kinds.  SMALL: per-CTA tables in shared memory ([S] counts, [S] first positions
// relative to the CTA's residue range), merged into the global tables with S atomics per CTA.  !SMALL: the
// tables are large and L2-resident; windows update them directly (low contention because S is large).
// ORDER = order-only mode (min_filter == 0 callers that do not need occurrence counts): no count table, and the launch
// is one CHUNK of a front-to-back walk over the shard — `state[0]` is the device-side "every code of the space has a
// first position" flag: CTAs of later chunks see it and return at once, and the last CTA of a chunk (ticket in
// state[1]) re-evaluates it.  first[c] of a code is final as soon as it is set by a chunk (chunks are walked in
// position order), so once all S codes are seen the rest of the shard cannot change the basis order.
template <bool SMALL, bool ORDER>
__global__ void __launch_bounds__(TS_THREADS) basis_kernel(const uint8_t *__restrict__ res, int64_t nres,
                                                           const int64_t *__restrict__ off, int64_t nseq,
                                                           const uint8_t *__restrict__ lut, uint32_t nsym, int k,
                                                           uint32_t pow_k1, int S, uint64_t res_base,
                                                           unsigned long long *__restrict__ g_count,
                                                           unsigned long long *__restrict__ g_first,
                                                           int *__restrict__ state) {
    extern __shared__ __align__(128) uint8_t s_raw[];   // symbol buffer, then (SMALL) the two tables
    __shared__ uint8_t s_lut[256];
    __shared__ int64_t s_range[2];
    __shared__ unsigned int s_nstart;
    __shared__ int s_flag;
    if (ORDER) {
        if (threadIdx.x == 0) s_flag = *reinterpret_cast<volatile int *>(state);
        __syncthreads();
        if (s_flag) return;                             // saturated by an earlier chunk: nothing left to learn
    }
    uint8_t *s_sym = s_raw;
    uint32_t *s_cnt = reinterpret_cast<uint32_t *>(s_raw + BS_SYM_BYTES), *s_min = ORDER ? s_cnt : s_cnt + S;
    uint32_t sym_addr = smem_addr(s_sym), cnt_addr = smem_addr(s_cnt), min_addr = smem_addr(s_min);
    asm volatile("" : "+r"(sym_addr), "+r"(cnt_addr), "+r"(min_addr));   // keep the window addresses in registers
    const int tid = threadIdx.x;
    ts_lut_init(s_lut, lut);
    if (SMALL) for (int i = tid; i < S; i += blockDim.x) { if (!ORDER) s_cnt[i] = 0; s_min[i] = 0xFFFFFFFFu; }
    if (tid == 0) { seq_range(off, nseq, blockIdx.x, gridDim.x, &s_range[0], &s_range[1]); s_nstart = 0; }
    __syncthreads();
    const int64_t lo = s_range[0], hi = s_range[1];
    const int64_t r_lo = (lo < hi) ? __ldg(off + lo) : 0, r_hi = (lo < hi) ? __ldg(off + hi) : 0;
    int64_t cur = lo;                 // first sequence that starts at or after `a`
    bool first = true;
    uint32_t tail = 0;
    for (int64_t a = r_lo; a < r_hi;) {
        const int64_t b = min(r_hi, (a + BS_SEG) & ~int64_t(15));
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
        if (mine) atomicAdd(&s_nstart, mine);
        __syncthreads();
        cur += s_nstart;
        const int C = ts_chunk(g.hi - g.lo);
        const int i0 = g.lo + tid * C, i1 = min(i0 + C, g.hi);
        // position of a window start relative to r_lo = shared address of its LAST symbol + to_rel
        const int64_t to_rel64 = (g.base - r_lo) - TS_PAD - (k - 1) - int64_t(sym_addr);
        const uint32_t to_rel = uint32_t(to_rel64);     // modular: the sum is in [0, 2^32)
        ts_scan_chunk<uint32_t>(
            sym_addr, i0, i1, k, nsym, pow_k1,
            [&](uint32_t p, uint32_t code, bool ok) {
                if (ok) {
                    const uint32_t rel = p + to_rel;
                    if (SMALL) {
                        if (!ORDER) reds_add_u32(cnt_addr + (code << 2), 1u);
                        if (rel < s_min[code]) reds_min_u32(min_addr + (code << 2), rel);
                    } else {
                        atomicAdd(g_count + code, 1ull);
                        const unsigned long long pos = res_base + uint64_t(r_lo) + rel;
                        // stale reads can only be too large (first is monotone decreasing): never skips a needed min
                        if (g_first && pos < __ldcg(g_first + code)) atomicMin(g_first + code, pos);
                    }
                }
            },
            [](uint32_t) {});
        tail = ts_tail_read(s_sym, g, k);
        first = false;
        a = b;
        __syncthreads();
        if (tid == 0) s_nstart = 0;    // ordered before the next atomicAdd by the barrier after staging
    }
    if (SMALL && lo < hi) {
        for (int i = tid; i < S; i += blockDim.x) {
            if (ORDER) {
                const uint32_t m = s_min[i];
                if (m != 0xFFFFFFFFu) atomicMin(g_first + i, (unsigned long long)(res_base + uint64_t(r_lo) + m));
            } else {
                const uint32_t c = s_cnt[i];
                if (c) {
                    atomicAdd(g_count + i, (unsigned long long)c);
                    if (g_first) atomicMin(g_first + i, (unsigned long long)(res_base + uint64_t(r_lo) + s_min[i]));
                }
            }
        }
    }
    if (ORDER) {
        // the last CTA of this chunk to get here counts the codes that have a first position
        __threadfence();
        __syncthreads();
        if (tid == 0) s_flag = (atomicAdd(state + 1, 1) == int(gridDim.x) - 1);
        __syncthreads();
        if (!s_flag) return;
        __threadfence();
        int seen = 0;
        for (int i = tid; i < S; i += blockDim.x) seen += (__ldcg(g_first + i) != ~0ull);
        __shared__ int s_seen;
        if (tid == 0) s_seen = 0;
        __syncthreads();
        if (seen) atomicAdd(&s_seen, seen);
        __syncthreads();
        if (tid == 0) {
            state[1] = 0;                               // ticket ready for the next chunk's launch
            state[2] = s_seen;
            if (s_seen == S) state[0] = 1;
            __threadfence();
        }
    }
}

__global__ void basis_keys_kernel(const uint64_t *__restrict__ count, const uint64_t *__restrict__ first, int64_t S,
                                  uint64_t min_filter, uint64_t *__restrict__ keys, uint64_t *__restrict__ vals) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < S; i += int64_t(gridDim.x) * blockDim.x) {
        keys[i] = (count ? count[i] > min_filter : true) ? first[i] : ~0ull;     // no counts: every code that was seen
        vals[i] = uint64_t(i);
    }
}

// after the sort: kept codes come first, ordered by first occurrence
__global__ void basis_emit_kernel(const uint64_t *__restrict__ keys_sorted, const uint64_t *__restrict__ codes_sorted,
                                  const uint64_t *__restrict__ count, int64_t S, uint64_t *__restrict__ basis_codes,
                                  uint64_t *__restrict__ basis_counts, int32_t *__restrict__ col_of_code,
                                  int64_t *__restrict__ K_out) {
    for (int64_t j = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; j < S; j += int64_t(gridDim.x) * blockDim.x) {
        const uint64_t key = keys_sorted[j], code = codes_sorted[j];
        const bool kept = key != ~0ull;
        if (kept) {
            basis_codes[j] = code;
            if (basis_counts) basis_counts[j] = count[code];
            if (col_of_code) col_of_code[code] = (int32_t)j;
            const bool last = (j + 1 == S) || (keys_sorted[j + 1] == ~0ull);
            if (last) *K_out = j + 1;
        } else {
            if (col_of_code) col_of_code[code] = -1;
            if (j == 0) *K_out = 0;
        }
    }
}

__global__ void colmap_fill_kernel(int32_t *col, int64_t S) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < S; i += int64_t(gridDim.x) * blockDim.x) col[i] = -1;
}
__global__ void colmap_scatter_kernel(const uint64_t *__restrict__ codes, int64_t K, int64_t S, int32_t *col) {
    for (int64_t j = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; j < K; j += int64_t(gridDim.x) * blockDim.x) {
        const uint64_t c = codes[j];
        if (c < (uint64_t)S) col[c] = (int32_t)j;
    }
}


// CTAs of a basis_kernel launch over nres residues with `smem` bytes of dynamic shared memory each
static int64_t basis_grid(int64_t nres, size_t smem) {
    int per_sm = int((227 * 1024) / (smem + 1536));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    int64_t grid = int64_t(sm_count()) * per_sm;
    const int64_t min_grid = (nres >> 30) + 1;           // keep each CTA's residue range well below 2^32
    if (grid < min_grid) grid = min_grid;
    const int64_t max_grid = (nres + BS_SEG - 1) / BS_SEG;   // no point in CTAs with less than a segment
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    return grid;
}

}  // namespace skm

extern "C" {

int skm_basis_accumulate(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                         const uint8_t *d_lut, int nsym, int k, uint64_t res_base, uint64_t *d_count,
                         uint64_t *d_first, skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (S128 > (unsigned __int128)SKM_DENSE_MAX_SPACE) {
        set_error("skm_basis_accumulate: code space %d^%d exceeds the table limit 2^27 (use the sorted path)", nsym, k);
        return SKM_ERR_UNSUPPORTED;
    }
    if (!d_count) { set_error("skm_basis_accumulate: NULL table"); return SKM_ERR_INVALID; }     // d_first may be NULL: counts only
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!ts_supported(nsym, k)) { set_error("skm_basis_accumulate: nsym=%d k=%d outside the kernel envelope (nsym <= %d, k <= %d)", nsym, k, TS_MAX_NSYM, TS_MAX_K); return SKM_ERR_UNSUPPORTED; }
    const int64_t S = (int64_t)S128;
    cudaStream_t st = (cudaStream_t)stream;
    auto *cnt = reinterpret_cast<unsigned long long *>(d_count);
    auto *fst = reinterpret_cast<unsigned long long *>(d_first);
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    const bool small = S <= SMALL_S;
    const size_t smem = size_t(BS_SYM_BYTES) + (small ? size_t(S) * 8 : 0);
    const int64_t grid = basis_grid(nres, smem);
    if (small) {
        auto kern = basis_kernel<true, false>;
        SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)grid, TS_THREADS, smem, st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k, pow_k1, (int)S, res_base, cnt, fst, nullptr);
    } else {
        auto kern = basis_kernel<false, false>;
        kern<<<(unsigned)grid, TS_THREADS, smem, st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k, pow_k1, (int)S, res_base, cnt, fst, nullptr);
    }
    SKM_LAUNCH_CHECK("basis_accumulate");
    return SKM_OK;
}

int skm_basis_order_max_space(void) { return (int)skm::SMALL_S; }

int skm_basis_first_progressive(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets,
                                const int64_t *h_offsets, int64_t nseq, const uint8_t *d_lut, int nsym, int k,
                                uint64_t res_base, uint64_t *d_first, int32_t *d_state, int64_t first_chunk_res,
                                int growth, skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (S128 > (unsigned __int128)SMALL_S) {
        set_error("skm_basis_first_progressive: code space %d^%d exceeds %lld (use skm_basis_accumulate)", nsym, k, (long long)SMALL_S);
        return SKM_ERR_UNSUPPORTED;
    }
    if (!d_first || !d_state || (nseq > 0 && !h_offsets)) { set_error("skm_basis_first_progressive: NULL argument"); return SKM_ERR_INVALID; }
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!ts_supported(nsym, k)) { set_error("skm_basis_first_progressive: nsym=%d k=%d outside the kernel envelope", nsym, k); return SKM_ERR_UNSUPPORTED; }
    if (first_chunk_res <= 0) first_chunk_res = 4ll << 20;
    if (growth < 2) growth = 4;
    const int64_t S = (int64_t)S128;
    cudaStream_t st = (cudaStream_t)stream;
    auto *fst = reinterpret_cast<unsigned long long *>(d_first);
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    const size_t smem = size_t(BS_SYM_BYTES) + size_t(S) * 4;
    auto kern = basis_kernel<true, true>;
    SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // chunks of sequences, front to back: ~first_chunk_res residues, then `growth` times more each time
    int64_t s_lo = 0, want = first_chunk_res;
    while (s_lo < nseq) {
        const int64_t r_lo = h_offsets[s_lo];
        int64_t s_hi = nseq;
        if (h_offsets[nseq] - r_lo > want + want / 2) {          // otherwise the rest goes in one launch
            const int64_t *it = std::lower_bound(h_offsets + s_lo + 1, h_offsets + nseq, r_lo + want);
            s_hi = it - h_offsets;
        }
        const int64_t chunk_res = h_offsets[s_hi] - r_lo;
        if (chunk_res > 0) {
            const int64_t grid = basis_grid(chunk_res, smem);
            kern<<<(unsigned)grid, TS_THREADS, smem, st>>>(d_residues, nres, d_offsets + s_lo, s_hi - s_lo, d_lut, (uint32_t)nsym, k,
                                                           pow_k1, (int)S, res_base, nullptr, fst, d_state);
            SKM_LAUNCH_CHECK("basis_first_progressive");
        }
        s_lo = s_hi;
        want *= growth;
    }
    return SKM_OK;
}

size_t skm_basis_finalize_workspace(int64_t S) {
    using namespace skm;
    if (S <= 0) return 256;
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const uint64_t *)nullptr, (uint64_t *)nullptr,
                                    (const uint64_t *)nullptr, (uint64_t *)nullptr, (int64_t)S);
    return 4 * align256(size_t(S) * 8) + align256(temp) + 256;
}

int skm_basis_finalize(const uint64_t *d_count, const uint64_t *d_first, int64_t S, int64_t min_filter,
                       uint64_t *d_basis_codes, uint64_t *d_basis_counts, int32_t *d_col_of_code, int64_t *d_K,
                       void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (S <= 0 || S > SKM_DENSE_MAX_SPACE) { set_error("skm_basis_finalize: S=%lld out of range", (long long)S); return SKM_ERR_INVALID; }
    if (!d_first || !d_basis_codes || !d_K) { set_error("skm_basis_finalize: NULL argument"); return SKM_ERR_INVALID; }
    if (!d_count && (min_filter > 0 || d_basis_counts)) { set_error("skm_basis_finalize: without d_count only min_filter = 0 and no d_basis_counts"); return SKM_ERR_INVALID; }
    if (d_count && !d_basis_counts) { set_error("skm_basis_finalize: NULL d_basis_counts"); return SKM_ERR_INVALID; }
    if (min_filter < 0) min_filter = 0;   // count > negative is always true for present k-mers; absent ones (count 0) must stay out
    const size_t need = skm_basis_finalize_workspace(S);
    if (!workspace || workspace_bytes < need) { set_error("skm_basis_finalize: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t seg = align256(size_t(S) * 8);
    char *p = reinterpret_cast<char *>(workspace);
    p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(p) + 255) & ~uintptr_t(255));
    uint64_t *keys_in = (uint64_t *)p, *keys_out = (uint64_t *)(p + seg);
    uint64_t *vals_in = (uint64_t *)(p + 2 * seg), *vals_out = (uint64_t *)(p + 3 * seg);
    void *temp = p + 4 * seg;
    size_t temp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys_in, keys_out, vals_in, vals_out, S);
    const int grid = (int)std::min<int64_t>((S + 255) / 256, int64_t(sm_count()) * 8);
    basis_keys_kernel<<<grid, 256, 0, st>>>(d_count, d_first, S, (uint64_t)min_filter, keys_in, vals_in);
    SKM_LAUNCH_CHECK("basis_keys_kernel");
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, vals_in, vals_out, S, 0, 64, st));
    basis_emit_kernel<<<grid, 256, 0, st>>>(keys_out, vals_out, d_count, S, d_basis_codes, d_basis_counts, d_col_of_code, d_K);
    SKM_LAUNCH_CHECK("basis_emit_kernel");
    return SKM_OK;
}

int skm_basis_colmap(const uint64_t *d_basis_codes, int64_t K, int64_t S, int32_t *d_col_of_code, skm_stream_t stream) {
    using namespace skm;
    if (S <= 0 || S > SKM_DENSE_MAX_SPACE || K < 0 || !d_col_of_code || (K > 0 && !d_basis_codes)) { set_error("skm_basis_colmap: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (int)std::min<int64_t>((S + 255) / 256, int64_t(sm_count()) * 8);
    colmap_fill_kernel<<<grid, 256, 0, st>>>(d_col_of_code, S);
    SKM_LAUNCH_CHECK("colmap_fill_kernel");
    if (K > 0) {
        const int g2 = (int)std::min<int64_t>((K + 255) / 256, int64_t(sm_count()) * 8);
        colmap_scatter_kernel<<<g2, 256, 0, st>>>(d_basis_codes, K, S, d_col_of_code);
        SKM_LAUNCH_CHECK("colmap_scatter_kernel");
    }
    return SKM_OK;
}

}  // extern "C"
