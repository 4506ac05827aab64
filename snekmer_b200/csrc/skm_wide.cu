// skm_wide.cu — vectorisation over code spaces too large for tables (nsym^k > 2^27, up to 2^64 - 1):
// the C5 sweep shapes (20 letters, k = 14 => 20^14 = 1.6e18 codes).
//
// The reference builds the basis as a dict of k-mer strings in first-occurrence order
// (kmerize.smk:89-104) and counts windows per sequence (learn.smk:359-383); neither needs a table
// over the code space.  Here both are sorts of 64-bit window codes:
//
//  skm_basis_sorted_local     one shard: code of every window (tile scanner, 64-bit rolling codes) paired with
//                             its position, radix-sorted by code over only the bits of nsym^k (stable, so the
//                             first element of a run is the first occurrence), run-length encoded into the
//                             table (code, count, first position + res_base) sorted by code.
//  skm_basis_sorted_finalize  one or more such tables (chunks of a shard, or the all-gathered tables of all
//                             GPUs): sort by code, reduce (sum of counts, min of first), drop count <=
//                             min_filter, order by first position => basis codes in the reference's order, plus
//                             the sorted code list with the column of every entry (the lookup structure).
//  skm_codes_to_columns       the code -> column lookup in the sorted code list.
// The per-sequence counts over a wide basis are skm_count_csr_sorted (skm_csrsort.cu) and its segmented-sort
// cross-check skm_count_csr_wide (skm_count.cu), which use wide_check and launch_window_codes64 from here.
// Everything is atomic-free and bit-reproducible.
#include <cub/cub.cuh>

#include "skm_common.cuh"
#include "skm_tile.cuh"

namespace skm {

constexpr int WD_SEG = ts_seg_cap(28);
constexpr int WD_SYM_BYTES = (ts_sym_bytes(WD_SEG) + 15) & ~15;
constexpr int WD_SMEM_BYTES = WD_SYM_BYTES + WD_SEG * 8;          // symbols + one staged 64-bit key per position
constexpr uint64_t WD_NONE = ~0ull;

// keys[p] = 64-bit code of the window whose LAST residue sits at position p, all-ones when invalid
__global__ void __launch_bounds__(TS_THREADS) window_codes64_kernel(const uint8_t *__restrict__ res, int64_t nres,
                                                                    const int64_t *__restrict__ off, int64_t nseq,
                                                                    const uint8_t *__restrict__ lut, uint64_t nsym, int k,
                                                                    uint64_t pow_k1, uint64_t *__restrict__ keys) {
    extern __shared__ __align__(128) uint8_t s_sym[];
    __shared__ uint8_t s_lut[256];
    __shared__ int64_t s_ctl[4];
    uint64_t *s_keys = reinterpret_cast<uint64_t *>(s_sym + WD_SYM_BYTES);
    ts_lut_init(s_lut, lut);
    __syncthreads();
    // keys are staged per segment and copied out coalesced (a thread's positions are 28 apart from its neighbour's)
    ts_range_scan_rows<uint64_t>(res, nres, off, nseq, s_lut, s_sym, WD_SEG, k, nsym, pow_k1, /*origin=*/0, s_ctl,
                                 [&](int64_t, int64_t, uint64_t code, bool ok, int local) { s_keys[local] = ok ? code : WD_NONE; },
                                 [&](int64_t rel_a, int n) {
                                     for (int i = threadIdx.x; i < n; i += blockDim.x) keys[rel_a + i] = s_keys[i];
                                 });
}

__global__ void __launch_bounds__(256) iota_u32_kernel(uint32_t *__restrict__ out, int64_t n) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) out[i] = uint32_t(i);
}

// after the run-length encode: first[r] = res_base + position of the first element of run r (the sort is stable);
// the run of the invalid key sorts last and is dropped
// (`first` may alias `starts`: element i reads its own start before it writes its own first position)
__global__ void __launch_bounds__(256) basis_runs_finish_kernel(const uint64_t *__restrict__ uniq, const int64_t *starts,
                                                                const uint32_t *__restrict__ pos_sorted,
                                                                const int64_t *__restrict__ num_runs, int64_t res_base,
                                                                int64_t *first, int64_t *__restrict__ n_out) {
    int64_t n = *num_runs;
    if (n > 0 && uniq[n - 1] == WD_NONE) --n;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
        first[i] = res_base + int64_t(pos_sorted[starts[i]]);
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = n;
}

__global__ void set_i64_kernel(int64_t *dst, int64_t v) { *dst = v; }
// dst[i] = v for i in [*n_ptr, n_cap)
__global__ void __launch_bounds__(256) pad_i64_kernel(int64_t *__restrict__ dst, const int64_t *__restrict__ n_ptr, int64_t n_cap, int64_t v) {
    for (int64_t i = *n_ptr + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_cap; i += int64_t(gridDim.x) * blockDim.x) dst[i] = v;
}

__global__ void __launch_bounds__(256) gather_i64_kernel(const int64_t *__restrict__ src, const uint32_t *__restrict__ idx, int64_t n,
                                                         int64_t *__restrict__ out) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) out[i] = src[idx[i]];
}

__global__ void __launch_bounds__(256) keep_flags_kernel(const int64_t *__restrict__ counts, const int64_t *__restrict__ n_ptr,
                                                         int64_t n_cap, int64_t min_filter, uint8_t *__restrict__ flags) {
    const int64_t n = *n_ptr;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_cap; i += int64_t(gridDim.x) * blockDim.x)
        flags[i] = (i < n && counts[i] > min_filter) ? 1 : 0;
}

// basis[c] = sorted_codes[order[c]], basis_counts[c] = counts[order[c]], col_of_sorted[order[c]] = c
__global__ void __launch_bounds__(256) basis_emit_kernel(const uint64_t *__restrict__ sorted_codes, const int64_t *__restrict__ counts,
                                                         const uint32_t *__restrict__ order, const int64_t *__restrict__ K_ptr,
                                                         uint64_t *__restrict__ basis, int64_t *__restrict__ basis_counts,
                                                         int32_t *__restrict__ col_of_sorted) {
    const int64_t K = *K_ptr;
    for (int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; c < K; c += int64_t(gridDim.x) * blockDim.x) {
        const uint32_t j = order[c];
        basis[c] = sorted_codes[j];
        if (basis_counts) basis_counts[c] = counts[j];
        col_of_sorted[j] = int32_t(c);
    }
}

__global__ void __launch_bounds__(256) codes_to_columns_kernel(const uint64_t *__restrict__ codes, int64_t n,
                                                               const uint64_t *__restrict__ sorted_codes,
                                                               const int32_t *__restrict__ col_of_sorted, int64_t K,
                                                               int32_t *__restrict__ cols) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
        cols[i] = lookup_column(sorted_codes, col_of_sorted, K, codes[i]);
}

struct MinI64 {
    __device__ __forceinline__ int64_t operator()(const int64_t &a, const int64_t &b) const { return a < b ? a : b; }
};

constexpr int64_t WD_MAX_RES = 1ll << 30;

// argument checks shared by the 64-bit entry points
int wide_check(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
                      int nsym, int k, const char *who, unsigned __int128 *S) {
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    if (!ts_supported(nsym, k)) { set_error("%s: nsym=%d k=%d outside the kernel envelope", who, nsym, k); return SKM_ERR_UNSUPPORTED; }
    code_space(nsym, k, S);
    if (*S > (((unsigned __int128)1 << 64) - 1)) { set_error("%s: nsym^k = 2^64 collides with the invalid sentinel", who); return SKM_ERR_UNSUPPORTED; }
    if (nres >= WD_MAX_RES || nseq >= (1ll << 31)) { set_error("%s: more than 2^30 residues per call; split the shard", who); return SKM_ERR_UNSUPPORTED; }
    return SKM_OK;
}

// keys[p] = 64-bit code of the window ending at position p (positions outside every sequence are left alone)
int launch_window_codes64(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
                                 int nsym, int k, uint64_t *d_keys, cudaStream_t st) {
    uint64_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint64_t)nsym;
    int64_t grid = int64_t(sm_count()) * 8;
    const int64_t max_grid = (nres + WD_SEG - 1) / WD_SEG;
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    SKM_CUDA_TRY(cudaFuncSetAttribute(window_codes64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WD_SMEM_BYTES));
    window_codes64_kernel<<<(unsigned)grid, TS_THREADS, WD_SMEM_BYTES, st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint64_t)nsym, k, pow_k1, d_keys);
    SKM_LAUNCH_CHECK("window_codes64_kernel");
    return SKM_OK;
}

}  // namespace skm

extern "C" {

size_t skm_basis_sorted_local_workspace(int64_t nres) {
    using namespace skm;
    if (nres <= 0) return 256;
    size_t t_sort = 0, t_rle = 0, t_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t_sort, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const uint32_t *)nullptr,
                                    (uint32_t *)nullptr, nres, 0, 64);
    cub::DeviceRunLengthEncode::Encode(nullptr, t_rle, (const uint64_t *)nullptr, (uint64_t *)nullptr, (int64_t *)nullptr,
                                       (int64_t *)nullptr, (int)std::min<int64_t>(nres, (1ll << 31) - 1));
    cub::DeviceScan::ExclusiveSum(nullptr, t_scan, (const int64_t *)nullptr, (int64_t *)nullptr, nres);
    return 2 * align256(size_t(nres) * 8) + 2 * align256(size_t(nres) * 4) + align256(std::max(t_sort, std::max(t_rle, t_scan))) + 1024;
}

int skm_basis_sorted_local(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                           const uint8_t *d_lut, int nsym, int k, int64_t res_base, uint64_t *d_codes_out,
                           int64_t *d_counts_out, int64_t *d_first_out, int64_t *d_n_out, void *workspace,
                           size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    unsigned __int128 S;
    int rc = wide_check(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, "skm_basis_sorted_local", &S);
    if (rc) return rc;
    if (!d_n_out) { set_error("skm_basis_sorted_local: d_n_out is NULL"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_n_out, 0, 8, st));
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!d_codes_out || !d_counts_out || !d_first_out) { set_error("skm_basis_sorted_local: NULL output"); return SKM_ERR_INVALID; }
    const size_t need = skm_basis_sorted_local_workspace(nres);
    if (!workspace || workspace_bytes < need) { set_error("skm_basis_sorted_local: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg8 = align256(size_t(nres) * 8), seg4 = align256(size_t(nres) * 4);
    uint64_t *keys_a = (uint64_t *)p, *keys_b = (uint64_t *)(p + seg8);
    uint32_t *pos_a = (uint32_t *)(p + 2 * seg8), *pos_b = (uint32_t *)(p + 2 * seg8 + seg4);
    void *temp = p + 2 * seg8 + 2 * seg4;
    size_t temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    const int grid = (int)std::min<int64_t>((nres + 255) / 256, int64_t(sm_count()) * 16);
    SKM_CUDA_TRY(cudaMemsetAsync(keys_a, 0xFF, size_t(nres) * 8, st));     // positions outside every sequence
    rc = launch_window_codes64(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, keys_a, st);
    if (rc) return rc;
    iota_u32_kernel<<<grid, 256, 0, st>>>(pos_a, nres);
    SKM_LAUNCH_CHECK("iota_u32_kernel");
    // valid codes are < S <= 2^end_bit - 1 = the low bits of the all-ones key, which therefore still sorts last
    const int end_bit = bits_for(S + 1);
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_a, keys_b, pos_a, pos_b, nres, 0, end_bit, st));
    int64_t *num_runs = reinterpret_cast<int64_t *>(keys_a);                // keys_a is free after the sort
    temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceRunLengthEncode::Encode(temp, temp_bytes, keys_b, d_codes_out, d_counts_out, num_runs, (int)nres, st));
    // run starts = exclusive sum of the run lengths, written to d_first_out and converted in place (element i
    // reads its own start and writes its own first position).  The scan covers all nres slots of d_counts_out:
    // the slots past the last run are zeroed first so that the scan reads defined values.
    pad_i64_kernel<<<grid, 256, 0, st>>>(d_counts_out, num_runs, nres, 0);
    SKM_LAUNCH_CHECK("pad_i64_kernel");
    temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, d_counts_out, d_first_out, nres, st));
    basis_runs_finish_kernel<<<grid, 256, 0, st>>>(d_codes_out, d_first_out, pos_b, num_runs, res_base, d_first_out, d_n_out);
    SKM_LAUNCH_CHECK("basis_runs_finish_kernel");
    return SKM_OK;
}

size_t skm_basis_sorted_finalize_workspace(int64_t n) {
    using namespace skm;
    if (n <= 0) return 256;
    size_t t = 0, t2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const uint32_t *)nullptr,
                                    (uint32_t *)nullptr, n, 0, 64);
    cub::DeviceReduce::ReduceByKey(nullptr, t2, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const int64_t *)nullptr,
                                   (int64_t *)nullptr, (int64_t *)nullptr, cub::Sum(), n);
    t = std::max(t, t2);
    cub::DeviceReduce::ReduceByKey(nullptr, t2, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const int64_t *)nullptr,
                                   (int64_t *)nullptr, (int64_t *)nullptr, MinI64(), n);
    t = std::max(t, t2);
    cub::DeviceSelect::Flagged(nullptr, t2, (const uint64_t *)nullptr, (const uint8_t *)nullptr, (uint64_t *)nullptr, (int64_t *)nullptr, n);
    t = std::max(t, t2);
    // keys_a keys_b (u64) | v1 v2 v3 (i64) | idx_a idx_b (u32) | flags (u8) | temp
    return 5 * align256(size_t(n) * 8) + 2 * align256(size_t(n) * 4) + align256(size_t(n)) + align256(t) + 1024;
}

int skm_basis_sorted_finalize(const uint64_t *d_codes, const int64_t *d_counts, const int64_t *d_first, int64_t n,
                              int merged, int64_t min_filter, int64_t first_bound, uint64_t *d_basis_out, int64_t *d_basis_counts_out,
                              uint64_t *d_sorted_codes_out, int32_t *d_col_of_sorted_out, int64_t *d_K_out,
                              void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (n < 0 || !d_K_out) { set_error("skm_basis_sorted_finalize: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_K_out, 0, 8, st));
    if (n == 0) return SKM_OK;
    if (n >= (1ll << 31)) { set_error("skm_basis_sorted_finalize: more than 2^31 table entries"); return SKM_ERR_UNSUPPORTED; }
    if (!d_codes || !d_counts || !d_first || !d_basis_out || !d_sorted_codes_out || !d_col_of_sorted_out) { set_error("skm_basis_sorted_finalize: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_basis_sorted_finalize_workspace(n);
    if (!workspace || workspace_bytes < need) { set_error("skm_basis_sorted_finalize: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg8 = align256(size_t(n) * 8), seg4 = align256(size_t(n) * 4);
    uint64_t *keys_a = (uint64_t *)p, *keys_b = (uint64_t *)(p + seg8);
    int64_t *v1 = (int64_t *)(p + 2 * seg8), *v2 = (int64_t *)(p + 3 * seg8), *v3 = (int64_t *)(p + 4 * seg8);
    uint32_t *idx_a = (uint32_t *)(p + 5 * seg8), *idx_b = (uint32_t *)(p + 5 * seg8 + seg4);
    uint8_t *flags = (uint8_t *)(p + 5 * seg8 + 2 * seg4);
    void *temp = p + 5 * seg8 + 2 * seg4 + align256(size_t(n));
    const size_t temp_cap = workspace_bytes - size_t((char *)temp - (char *)workspace);
    size_t temp_bytes;
    const int grid = (int)std::min<int64_t>((n + 255) / 256, int64_t(sm_count()) * 16);
    int64_t *d_m = d_K_out;      // number of distinct codes; overwritten by K in step 3

    // ---- 1. one entry per code, sorted by code: (code, sum of counts, min of first) ----
    const uint64_t *codes_m = d_codes;
    const int64_t *counts_m = d_counts, *first_m = d_first;
    if (merged) {
        set_i64_kernel<<<1, 1, 0, st>>>(d_m, n);
        SKM_LAUNCH_CHECK("set_i64_kernel");
    } else {
        iota_u32_kernel<<<grid, 256, 0, st>>>(idx_a, n);
        SKM_LAUNCH_CHECK("iota_u32_kernel");
        temp_bytes = temp_cap;
        SKM_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, d_codes, keys_a, idx_a, idx_b, n, 0, 64, st));
        gather_i64_kernel<<<grid, 256, 0, st>>>(d_counts, idx_b, n, v1);
        SKM_LAUNCH_CHECK("gather_i64_kernel");
        gather_i64_kernel<<<grid, 256, 0, st>>>(d_first, idx_b, n, v2);
        SKM_LAUNCH_CHECK("gather_i64_kernel");
        temp_bytes = temp_cap;
        SKM_CUDA_TRY(cub::DeviceReduce::ReduceByKey(temp, temp_bytes, keys_a, keys_b, v1, v3, d_m, cub::Sum(), n, st));
        temp_bytes = temp_cap;
        SKM_CUDA_TRY(cub::DeviceReduce::ReduceByKey(temp, temp_bytes, keys_a, d_sorted_codes_out /* scratch */, v2, v1, d_m, MinI64(), n, st));
        codes_m = keys_b; counts_m = v3; first_m = v1;       // free now: keys_a, v2, idx_a, idx_b
    }
    // ---- 2. min_filter: keep count > min_filter (kmerize.smk:97-104) ----
    const int64_t *cnt_sel, *first_sel;
    if (merged && min_filter <= 0) {
        // one merged table and nothing to filter (every entry occurs at least once): K = n, no selection passes
        cnt_sel = counts_m;
        first_sel = first_m;
        SKM_CUDA_TRY(cudaMemcpyAsync(d_sorted_codes_out, codes_m, size_t(n) * 8, cudaMemcpyDeviceToDevice, st));
    } else {
        keep_flags_kernel<<<grid, 256, 0, st>>>(counts_m, d_m, n, min_filter, flags);
        SKM_LAUNCH_CHECK("keep_flags_kernel");
        int64_t *cnt_w = v2, *first_w = reinterpret_cast<int64_t *>(keys_a);
        int64_t *d_tmpK = reinterpret_cast<int64_t *>(idx_a);    // two throw-away selection counts
        temp_bytes = temp_cap;
        SKM_CUDA_TRY(cub::DeviceSelect::Flagged(temp, temp_bytes, counts_m, flags, cnt_w, d_tmpK, n, st));
        temp_bytes = temp_cap;
        SKM_CUDA_TRY(cub::DeviceSelect::Flagged(temp, temp_bytes, first_m, flags, first_w, d_tmpK, n, st));
        temp_bytes = temp_cap;
        SKM_CUDA_TRY(cub::DeviceSelect::Flagged(temp, temp_bytes, codes_m, flags, d_sorted_codes_out, d_K_out, n, st));   // d_m dead from here
        // padding behind the K kept entries sorts last in step 3
        pad_i64_kernel<<<grid, 256, 0, st>>>(first_w, d_K_out, n, INT64_MAX);
        SKM_LAUNCH_CHECK("pad_i64_kernel");
        cnt_sel = cnt_w;
        first_sel = first_w;
    }
    // ---- 3. first-occurrence order: sort the kept entries by first position ----
    iota_u32_kernel<<<grid, 256, 0, st>>>(idx_a, n);
    SKM_LAUNCH_CHECK("iota_u32_kernel");
    temp_bytes = temp_cap;
    // positions are < first_bound <= 2^end_bit - 1 = the low bits of the padding value, which therefore still sorts last
    const int order_bits = first_bound > 0 ? bits_for((unsigned __int128)first_bound + 1) : 64;
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, reinterpret_cast<const uint64_t *>(first_sel), keys_b, idx_a, idx_b, n, 0, order_bits, st));
    basis_emit_kernel<<<grid, 256, 0, st>>>(d_sorted_codes_out, cnt_sel, idx_b, d_K_out, d_basis_out, d_basis_counts_out, d_col_of_sorted_out);
    SKM_LAUNCH_CHECK("basis_emit_kernel");
    return SKM_OK;
}

int skm_codes_to_columns(const uint64_t *d_codes, int64_t n, const uint64_t *d_sorted_codes, const int32_t *d_col_of_sorted,
                         int64_t K, int32_t *d_cols_out, skm_stream_t stream) {
    using namespace skm;
    if (n < 0 || K < 0) { set_error("skm_codes_to_columns: negative size"); return SKM_ERR_INVALID; }
    if (n == 0) return SKM_OK;
    if (!d_codes || !d_cols_out || (K > 0 && (!d_sorted_codes || !d_col_of_sorted))) { set_error("skm_codes_to_columns: NULL argument"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>((n + 255) / 256, int64_t(sm_count()) * 16);
    codes_to_columns_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_codes, n, d_sorted_codes, d_col_of_sorted, K, d_cols_out);
    SKM_LAUNCH_CHECK("codes_to_columns_kernel");
    return SKM_OK;
}

}  // extern "C"
