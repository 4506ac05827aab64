// skm_rows.cu — learn (c) for the heavy annotations of a Zipf-distributed family-size distribution: dense count rows.
//
// The sort-based sparse learn (skm_sparse.cu) moves ~40 bytes per window through radix-sort passes.  Family sizes are
// heavy-tailed (learn.smk's inputs are protein families: a few annotations own most sequences), and an annotation with
// more windows than about a quarter of the code space S is better counted than sorted: its row of S counters (6.7 MB
// for the 6-letter k = 8 space) stays in the 126 MB L2 while its sequences — gathered together — stream past, one
// 32-bit integer atomic per window, and the row read in code order IS the sorted run-length-encoded list.  The
// unannotated sequences get a row of their own, so the Totals row of learn.smk:380 is the column sum of all rows plus
// the column sums of the sorted (light) part: no separate pass over the residues.
//   skm_rows_accumulate    rows[row_of_seq[s]][code] += 1 for every valid window (sequences with row < 0 are skipped)
//   skm_rows_block_counts  non-zeros per (row, 4096-code block): the caller's prefix sums give every block its place
//   skm_rows_emit          (annotation * S + code, count) of every non-zero, in order, at the block's place
//   skm_rows_colsum        totals[c] += sum over rows of rows[r][c]
// Integer adds only: results are order-independent, hence bit-reproducible and equal to the sorted path's.
#include "skm_common.cuh"
#include "skm_tile.cuh"

namespace skm {

constexpr int RW_SEG = ts_seg_cap(28);                     // 7168 positions per staged segment
constexpr int RW_SYM_BYTES = (ts_sym_bytes(RW_SEG) + 15) & ~15;
constexpr int RW_BLOCK = 4096;                             // codes per compaction block

__global__ void __launch_bounds__(TS_THREADS) rows_accumulate_kernel(const uint8_t *__restrict__ res, int64_t nres,
                                                                     const int64_t *__restrict__ off, int64_t nseq,
                                                                     const uint8_t *__restrict__ lut, uint32_t nsym, int k,
                                                                     uint32_t pow_k1, const int32_t *__restrict__ row_of_seq,
                                                                     uint64_t S, uint32_t *__restrict__ rows) {
    extern __shared__ __align__(128) uint8_t s_sym[];
    __shared__ uint8_t s_lut[256];
    __shared__ int64_t s_ctl[4];
    ts_lut_init(s_lut, lut);
    __syncthreads();
    int64_t cur_row = -2;
    uint32_t *base = nullptr;
    ts_range_scan_rows<uint32_t>(res, nres, off, nseq, s_lut, s_sym, RW_SEG, k, nsym, pow_k1, /*origin=*/0, s_ctl,
                                 [&](int64_t, int64_t row, uint32_t code, bool ok, int) {
                                     if (!ok) return;
                                     if (row != cur_row) {
                                         cur_row = row;
                                         const int32_t r = __ldg(row_of_seq + row);
                                         base = r >= 0 ? rows + uint64_t(r) * S : nullptr;
                                     }
                                     if (base) atomicAdd(base + code, 1u);
                                 },
                                 [](int64_t, int) {});
}

// grid = (blocks per row, rows): non-zeros of rows[r][b * RW_BLOCK ...)
__global__ void __launch_bounds__(256) rows_block_counts_kernel(const uint32_t *__restrict__ rows, int64_t S, int nblk,
                                                                int32_t *__restrict__ counts) {
    const int b = blockIdx.x, r = blockIdx.y;
    const uint32_t *row = rows + uint64_t(r) * uint64_t(S);
    const int64_t c0 = int64_t(b) * RW_BLOCK, c1 = (c0 + RW_BLOCK < S) ? c0 + RW_BLOCK : S;
    int n = 0;
    for (int64_t c = c0 + threadIdx.x; c < c1; c += blockDim.x) n += (__ldg(row + c) != 0u);
    __shared__ int s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    if (n) atomicAdd(&s_n, n);
    __syncthreads();
    if (threadIdx.x == 0) counts[int64_t(r) * nblk + b] = s_n;
}

// grid as above; block (r, b) writes its non-zeros, in code order, from dst_row[r] + blk_off[r * nblk + b]
__global__ void __launch_bounds__(256) rows_emit_kernel(const uint32_t *__restrict__ rows, int64_t S, int nblk,
                                                        const int64_t *__restrict__ blk_off, const int64_t *__restrict__ dst_row,
                                                        const int64_t *__restrict__ ann_of_row, uint64_t *__restrict__ keys_out,
                                                        int64_t *__restrict__ vals_out, int64_t capacity) {
    const int b = blockIdx.x, r = blockIdx.y, t = threadIdx.x;
    const uint32_t *row = rows + uint64_t(r) * uint64_t(S);
    const int64_t c0 = int64_t(b) * RW_BLOCK;
    constexpr int PER = RW_BLOCK / 256;                     // consecutive codes per thread
    uint32_t v[PER];
    int mine = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int64_t c = c0 + int64_t(t) * PER + j;
        v[j] = c < S ? __ldg(row + c) : 0u;
        mine += (v[j] != 0u);
    }
    // exclusive scan of `mine` over the 256 threads
    __shared__ int s_warp[8];
    const int lane = t & 31, w = t >> 5;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int x = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += x; }
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    int before = 0;
    for (int i = 0; i < w; ++i) before += s_warp[i];
    int64_t pos = dst_row[r] + blk_off[int64_t(r) * nblk + b] + before + (incl - mine);
    const uint64_t key0 = uint64_t(ann_of_row[r]) * uint64_t(S) + uint64_t(c0) + uint64_t(t) * PER;
#pragma unroll
    for (int j = 0; j < PER; ++j)
        if (v[j] != 0u) {
            if (pos < capacity) { keys_out[pos] = key0 + j; vals_out[pos] = int64_t(v[j]); }
            ++pos;
        }
}

__global__ void __launch_bounds__(256) rows_colsum_kernel(const uint32_t *__restrict__ rows, int64_t S, int n_rows,
                                                          unsigned long long *__restrict__ totals) {
    for (int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; c < S; c += int64_t(gridDim.x) * blockDim.x) {
        unsigned long long t = 0;
        for (int r = 0; r < n_rows; ++r) t += __ldg(rows + uint64_t(r) * uint64_t(S) + c);
        if (t) totals[c] += t;
    }
}

}  // namespace skm

extern "C" {

int skm_rows_accumulate(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
                        int nsym, int k, const int32_t *d_row_of_seq, int64_t S, uint32_t *d_rows, skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (S128 > (unsigned __int128)SKM_DENSE_MAX_SPACE || (int64_t)S128 != S) { set_error("skm_rows_accumulate: S must equal nsym^k and be <= 2^27"); return SKM_ERR_UNSUPPORTED; }
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!d_row_of_seq || !d_rows) { set_error("skm_rows_accumulate: NULL argument"); return SKM_ERR_INVALID; }
    if (!ts_supported(nsym, k)) { set_error("skm_rows_accumulate: nsym=%d k=%d outside the kernel envelope", nsym, k); return SKM_ERR_UNSUPPORTED; }
    if (nres >= (1ll << 32)) { set_error("skm_rows_accumulate: more than 2^32 residues per call (32-bit counters); split the shard"); return SKM_ERR_UNSUPPORTED; }
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    int64_t grid = int64_t(sm_count()) * 8;
    const int64_t max_grid = (nres + RW_SEG - 1) / RW_SEG;
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    rows_accumulate_kernel<<<(unsigned)grid, TS_THREADS, RW_SYM_BYTES, (cudaStream_t)stream>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k,
                                                                                              pow_k1, d_row_of_seq, (uint64_t)S, d_rows);
    SKM_LAUNCH_CHECK("rows_accumulate_kernel");
    return SKM_OK;
}

int skm_rows_block(void) { return skm::RW_BLOCK; }

int skm_rows_block_counts(const uint32_t *d_rows, int64_t n_rows, int64_t S, int32_t *d_counts, skm_stream_t stream) {
    using namespace skm;
    if (n_rows < 0 || S <= 0 || n_rows > 65535) { set_error("skm_rows_block_counts: bad sizes (at most 65535 rows)"); return SKM_ERR_INVALID; }
    if (n_rows == 0) return SKM_OK;
    if (!d_rows || !d_counts) { set_error("skm_rows_block_counts: NULL argument"); return SKM_ERR_INVALID; }
    const int nblk = int((S + RW_BLOCK - 1) / RW_BLOCK);
    rows_block_counts_kernel<<<dim3(nblk, (unsigned)n_rows), 256, 0, (cudaStream_t)stream>>>(d_rows, S, nblk, d_counts);
    SKM_LAUNCH_CHECK("rows_block_counts_kernel");
    return SKM_OK;
}

int skm_rows_emit(const uint32_t *d_rows, int64_t n_rows, int64_t S, const int64_t *d_block_offsets, const int64_t *d_row_dst,
                  const int64_t *d_ann_of_row, uint64_t *d_keys_out, int64_t *d_vals_out, int64_t out_capacity, skm_stream_t stream) {
    using namespace skm;
    if (n_rows < 0 || S <= 0 || n_rows > 65535 || out_capacity < 0) { set_error("skm_rows_emit: bad sizes"); return SKM_ERR_INVALID; }
    if (n_rows == 0) return SKM_OK;
    if (!d_rows || !d_block_offsets || !d_row_dst || !d_ann_of_row || !d_keys_out || !d_vals_out) { set_error("skm_rows_emit: NULL argument"); return SKM_ERR_INVALID; }
    const int nblk = int((S + RW_BLOCK - 1) / RW_BLOCK);
    rows_emit_kernel<<<dim3(nblk, (unsigned)n_rows), 256, 0, (cudaStream_t)stream>>>(d_rows, S, nblk, d_block_offsets, d_row_dst, d_ann_of_row, d_keys_out,
                                                                                    d_vals_out, out_capacity);
    SKM_LAUNCH_CHECK("rows_emit_kernel");
    return SKM_OK;
}

int skm_rows_colsum(const uint32_t *d_rows, int64_t n_rows, int64_t S, int64_t *d_totals, skm_stream_t stream) {
    using namespace skm;
    if (n_rows < 0 || S <= 0 || n_rows > (1 << 30)) { set_error("skm_rows_colsum: bad sizes"); return SKM_ERR_INVALID; }
    if (n_rows == 0) return SKM_OK;
    if (!d_rows || !d_totals) { set_error("skm_rows_colsum: NULL argument"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>((S + 255) / 256, int64_t(sm_count()) * 16);
    rows_colsum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_rows, S, (int)n_rows, reinterpret_cast<unsigned long long *>(d_totals));
    SKM_LAUNCH_CHECK("rows_colsum_kernel");
    return SKM_OK;
}

}  // extern "C"
