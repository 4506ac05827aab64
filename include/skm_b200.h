/*
 * skm_b200.h — C ABI of the B200-native Snekmer hot path (libskm_b200.so).
 *
 * The reference (PNNL-CompBio/Snekmer 1.3.0) is pure Python and has no FFI; the
 * boundary it exposes is the Python module API (snekmer.vectorize.KmerVec,
 * snekmer.alphabet, snekmer.io) and the rule-body loops in the snekmer/rules .smk files.
 * Each entry point below names the reference code it replaces (file:line under
 * /root/reference).  The Python package snekmer_b200 binds these with ctypes
 * (snekmer_b200/_native.py); INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types in any signature;
 *   - every d_* pointer is DEVICE memory owned by the caller; the library never
 *     allocates persistent device memory; scratch comes from the caller through
 *     (workspace, workspace_bytes) sized by the matching *_workspace() query;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*)
 *     and re-entrant; no call synchronises the device unless stated;
 *   - return 0 on success, a negative SKM_ERR_* otherwise; skm_last_error()
 *     returns a thread-local message for the last failure;
 *   - sequences are a packed byte buffer `d_residues[nres]` (ASCII, base
 *     pointer 16-byte aligned) plus `d_offsets[nseq+1]` (int64, offsets[0]=0 is
 *     not required: offsets are positions in d_residues);
 *   - k-mer codes: code = sum_i sym_i * nsym^(k-1-i) with sym_i the index of
 *     the reduced symbol in the *sorted* output-symbol string; nsym^k <= 2^64.
 */
#ifndef SKM_B200_H
#define SKM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(SKM_BUILDING)
#define SKM_API __attribute__((visibility("default")))
#else
#define SKM_API
#endif

#define SKM_OK 0
#define SKM_ERR_INVALID (-1)     /* bad argument */
#define SKM_ERR_CUDA (-2)        /* CUDA runtime error (message has the string) */
#define SKM_ERR_UNSUPPORTED (-3) /* valid request outside the built envelope */
#define SKM_ERR_WORKSPACE (-4)   /* workspace too small */

#define SKM_INVALID_SYMBOL 0xFF
#define SKM_DENSE_MAX_SPACE (1ll << 27) /* largest nsym^k handled by table kernels */

typedef void *skm_stream_t; /* cudaStream_t */

/* library / device ------------------------------------------------------- */
SKM_API int skm_version(void);
SKM_API const char *skm_last_error(void);
/* sm_count, compute capability of the current device */
SKM_API int skm_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* (a1) residue -> symbol LUT.  Replaces the dict lookups of
 * alphabet.py:88-96 (FULL_ALPHABETS) + vectorize.py:193-195 (translate) +
 * vectorize.py:247 (char_set test).  map_from[i] -> map_to[i] for i < nmap;
 * symbols = sorted output symbols.  A byte is valid iff its translated
 * character is one of `symbols` (unmapped bytes translate to themselves).
 * Host-only, no CUDA. */
SKM_API int skm_lut_build(const char *map_from, const char *map_to, int nmap,
                  const char *symbols, int nsym, uint8_t lut_out[256]);

/* (a3) reduce(): vectorize.py:173-195 on the packed buffer — byte-wise
 * translate with a 256-entry char map (rstrip('*') is applied by the caller on
 * the offsets: it only shortens the strings). */
SKM_API int skm_reduce_bytes(const uint8_t *d_residues, int64_t nres,
                     const uint8_t *d_charmap, uint8_t *d_out,
                     skm_stream_t stream);

/* (a5/a6) KmerVec._kmer_gen / reduce_vectorize, vectorize.py:239-249,292-328:
 * code of the window starting at every residue position, or all-ones
 * (0xFFFFFFFF / 0xFFFFFFFFFFFFFFFF) where the window is invalid, crosses the
 * end of its sequence or the position belongs to no sequence.
 * code_bits = 32 requires nsym^k < 2^32, 64 requires nsym^k <= 2^64 - 1. */
SKM_API int skm_encode_windows(const uint8_t *d_residues, int64_t nres,
                       const int64_t *d_offsets, int64_t nseq,
                       const uint8_t *d_lut, int nsym, int k, int code_bits,
                       void *d_codes_out, skm_stream_t stream);

/* (a7) basis construction, kmerize.smk:89-104, pass 1 over the FASTA.
 * Accumulates into caller-initialised tables over the code space S = nsym^k
 * (S <= SKM_DENSE_MAX_SPACE): d_count[c] += occurrences (init 0),
 * d_first[c] = min(res_base + position of window start) (init all-ones).
 * res_base is the global residue position of d_residues[0] so that several
 * shards / GPUs can be merged by sum / min before skm_basis_finalize.
 * d_first may be NULL: occurrence counts only (the Totals row of learn.smk:380). */
SKM_API int skm_basis_accumulate(const uint8_t *d_residues, int64_t nres,
                         const int64_t *d_offsets, int64_t nseq,
                         const uint8_t *d_lut, int nsym, int k,
                         uint64_t res_base, uint64_t *d_count,
                         uint64_t *d_first, skm_stream_t stream);

/* (a7) order-only variant of pass 1 for min_filter = 0 (kmerize.smk:89-104 keeps every k-mer that
 * occurs, so the basis is fully determined by the first positions): the shard is walked front to
 * back in chunks of sequences (about first_chunk_res residues, then `growth` times more per chunk;
 * 0 = defaults) and the walk ends ON THE DEVICE as soon as every code of the space has a first
 * position — later chunks' CTAs return at once, no host synchronisation.  A space that never
 * saturates costs one full pass, like skm_basis_accumulate.  Code spaces up to
 * skm_basis_order_max_space() (shared-memory tables).  d_first as in skm_basis_accumulate (init
 * all-ones); d_state is int32[4], zero-initialised by the caller ([0] = saturated, [2] = codes
 * seen when last evaluated).  h_offsets is the HOST copy of d_offsets (chunk boundaries). */
SKM_API int skm_basis_order_max_space(void);
SKM_API int skm_basis_first_progressive(const uint8_t *d_residues, int64_t nres,
                                const int64_t *d_offsets, const int64_t *h_offsets,
                                int64_t nseq, const uint8_t *d_lut, int nsym, int k,
                                uint64_t res_base, uint64_t *d_first, int32_t *d_state,
                                int64_t first_chunk_res, int growth, skm_stream_t stream);

/* kmerize.smk:102-104 + dict insertion order: keep codes with
 * count > min_filter, order by first occurrence.  d_count and d_basis_counts may both be NULL
 * (order-only tables of skm_basis_first_progressive; min_filter must be 0): every code with a
 * first position is kept.  Writes d_basis_codes[0..K),
 * d_basis_counts[0..K), d_col_of_code[c] = column or -1 for every c < S, and K
 * to *d_K (device int64).  Capacity of the two basis arrays: S. */
SKM_API size_t skm_basis_finalize_workspace(int64_t S);
SKM_API int skm_basis_finalize(const uint64_t *d_count, const uint64_t *d_first,
                       int64_t S, int64_t min_filter, uint64_t *d_basis_codes,
                       uint64_t *d_basis_counts, int32_t *d_col_of_code,
                       int64_t *d_K, void *workspace, size_t workspace_bytes,
                       skm_stream_t stream);

/* kmerize.smk:72-78 (basis.txt branch) / learn on a given kmerlist:
 * d_col_of_code[c] = j for c = d_basis_codes[j], -1 elsewhere. */
SKM_API int skm_basis_colmap(const uint64_t *d_basis_codes, int64_t K, int64_t S,
                     int32_t *d_col_of_code, skm_stream_t stream);

/* (a9/a11) per-sequence k-mer counts over the basis, dense rows:
 * kmerize.smk:112-120 (presence = counts > 0), learn.smk:359-383,
 * apply.smk:195-206.  d_counts is [nseq, K] row-major; out_bits 32 (int32)
 * or 16 (uint16, requires max_len <= 65535).  d_col_of_code may be NULL for
 * the identity basis (column = code, K = S).  max_len = longest sequence
 * (0 = unknown: 32-bit shared-memory counters are used). */
SKM_API int skm_count_dense(const uint8_t *d_residues, int64_t nres,
                    const int64_t *d_offsets, int64_t nseq,
                    const uint8_t *d_lut, int nsym, int k,
                    const int32_t *d_col_of_code, int64_t S, int64_t K,
                    int out_bits, void *d_counts, int64_t max_len,
                    skm_stream_t stream);

/* same counts as CSR for large bases (learn.smk:359-383 at K ~ 1e6): per
 * sequence the sorted distinct columns (or codes when d_col_of_code is NULL;
 * nsym^k < 2^32) and their counts.  d_rowptr is int64 [nseq+1] (nnz =
 * d_rowptr[nseq]); d_cols / d_vals need capacity nres (an upper bound of nnz).
 * One call handles < 2^30 residues. */
SKM_API size_t skm_count_csr_workspace(int64_t nres, int64_t nseq);
SKM_API int skm_count_csr(const uint8_t *d_residues, int64_t nres,
                  const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
                  int nsym, int k, const int32_t *d_col_of_code, int64_t S,
                  int64_t *d_rowptr, uint32_t *d_cols, int32_t *d_vals,
                  void *workspace, size_t workspace_bytes,
                  skm_stream_t stream);

/* (a12/a13) learn: Library.filter_and_construct + _process_annotation_counts,
 * learn.smk:316-326,385-408, fused with the per-sequence counting of
 * learn.smk:359-383 (counts are never materialised):
 *   M[a,:]     = sum of the count rows of the sequences with d_ann_id[s] == a
 *   M[n_ann,:] = the same sum over sequences with d_ann_id[s] < 0 (unannotated,
 *                or the earlier copies of a duplicated id) — the "rest" row
 *   totals[:]  = column sum of all n_ann+1 rows = Totals over ALL sequences
 *                (learn.smk:380).
 * d_order (nullable) is a permutation of 0..nseq-1 that groups equal
 * annotation ids (a stable sort by id): each CTA then adds one shared-memory
 * row per run to M, so the reduction is contention-free and, being integer,
 * bit-reproducible.  d_M is int64 [n_ann+1, K], d_totals int64 [K]; both are
 * overwritten.  K*4 bytes must fit shared memory (K <= 51200). */
SKM_API int skm_learn_dense(const uint8_t *d_residues, int64_t nres,
                    const int64_t *d_offsets, int64_t nseq,
                    const uint8_t *d_lut, int nsym, int k,
                    const int32_t *d_col_of_code, int64_t S, int64_t K,
                    const int32_t *d_ann_id, const int64_t *d_order,
                    int64_t n_ann, int64_t *d_M, int64_t *d_totals,
                    skm_stream_t stream);

/* (a12/a13 at large K) learn, sparse: every valid window of a sequence with d_ann_id[s] >= 0
 * becomes the key ann * S + code (S = nsym^k < 2^32); keys are radix-sorted and run-length
 * encoded (no atomics).  Output: a COO list sorted by key — d_keys_out / d_vals_out need
 * capacity nres, the number of entries goes to *d_nnz (device int64).  Totals over all
 * sequences (learn.smk:380) are the counts of skm_basis_accumulate.  < 2^31 residues per call. */
SKM_API size_t skm_learn_sparse_workspace(int64_t nres);
SKM_API int skm_learn_sparse(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets,
                     int64_t nseq, const uint8_t *d_lut, int nsym, int k,
                     const int32_t *d_ann_id, int64_t n_ann, uint64_t *d_keys_out,
                     int64_t *d_vals_out, int64_t *d_nnz, void *workspace,
                     size_t workspace_bytes, skm_stream_t stream);

/* (a12 at large K, grouped) the same COO list built one annotation slice at a time with 32-bit keys.  The caller
 * gathers the sequences of annotations [ann_lo, ann_lo + ann_n) into one batch (skm_gather_sequences; unannotated
 * sequences never enter) with ann_n * nsym^k < 2^32 - 1; their (key, count) runs are appended at *d_nnz_inout
 * (device int64, read and advanced in stream order) as global keys ann * S + code.  Slices processed in annotation
 * order leave one sorted list.  Entries beyond out_capacity are dropped (check *d_nnz_inout <= capacity afterwards). */
SKM_API size_t skm_learn_sparse_group_workspace(int64_t nres);
SKM_API int skm_learn_sparse_group(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                           const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t ann_lo,
                           int64_t ann_n, uint64_t *d_keys_out, int64_t *d_vals_out, int64_t out_capacity,
                           int64_t *d_nnz_inout, void *workspace, size_t workspace_bytes, skm_stream_t stream);
/* skm_learn_sparse_group writing its entries straight into a LARGER sorted list that also holds blocks other paths produce
 * (the dense rows of heavy annotations, skm_rows_emit): block h belongs to annotation d_ins_ann[h] (ascending) and
 * d_ins_cum[h] is the inclusive prefix of the block sizes, so an entry of annotation a is stored d_ins_cum[#(ins_ann < a) - 1]
 * places further up (capacity counts the larger list).  d_ins_pos[h] (pre-set to INT64_MAX by the caller) receives the
 * smallest index of this list behind block h's predecessors: min over h' >= h, capped by the final *d_nnz_inout, is the
 * number of this list's entries in front of block h.  d_totals (nullable, int64 [S]) += count per code (learn.smk:380). */
SKM_API int skm_learn_sparse_group_place(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                                 const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t ann_lo, int64_t ann_n,
                                 uint64_t *d_keys_out, int64_t *d_vals_out, int64_t out_capacity, int64_t *d_nnz_inout,
                                 const int64_t *d_ins_ann, const int64_t *d_ins_cum, int64_t n_ins, int64_t *d_ins_pos, int64_t *d_totals,
                                 void *workspace, size_t workspace_bytes, skm_stream_t stream);
/* d_out_residues[d_out_offsets[i] ...] = sequence d_sel[i] of (d_residues, d_offsets): reorders / selects
 * sequences on the device (grouping by annotation, learn.smk:316-326 keeps only annotated sequences). */
SKM_API int skm_gather_sequences(const uint8_t *d_residues, const int64_t *d_offsets, const int64_t *d_sel,
                         int64_t n_sel, uint8_t *d_out_residues, const int64_t *d_out_offsets,
                         skm_stream_t stream);

/* Merge.merge_dataframes (learn.smk:467-494) for sparse matrices / fan-in of per-GPU lists:
 * entries with equal keys are summed; output sorted by key, capacity n, count in *d_n_out.
 * key_bound: exclusive upper bound of the keys (n_ann * S), 0 = unknown — limits the bits of the sort. */
SKM_API size_t skm_coo_merge_workspace(int64_t n);
SKM_API int skm_coo_merge(const uint64_t *d_keys_in, const int64_t *d_vals_in, int64_t n, uint64_t key_bound,
                  uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_n_out,
                  void *workspace, size_t workspace_bytes, skm_stream_t stream);

/* (a12/a13 at nsym^k beyond the tables, up to 2^64 - 1) learn, wide: learn.smk:306-326,359-408 with the matrix keyed by
 * BASIS COLUMN.  The basis is (d_sorted_codes uint64 [K] ascending, d_col_of_sorted int32 [K]: its column of each),
 * K < 2^31, as skm_basis_sorted_finalize gives it.  Every valid window whose code the basis holds becomes the key
 * a * K + col, with a = d_ann_id[s] when it is in [0, n_ann) and a = n_ann (the rest row) otherwise; keys are
 * radix-sorted and run-length encoded (no atomics).  Output: a COO list sorted by key, capacity nres, the number of
 * entries in *d_nnz (device int64).  The Totals row (learn.smk:380: occurrences over ALL sequences, restricted to the
 * basis columns) is skm_coo_colsum of the whole list with S = K; the annotated matrix is its prefix key < n_ann * K.
 * Needs (n_ann + 2) * K < 2^63.  One call handles < 2^30 residues: split larger shards and merge the chunks' sorted
 * lists with skm_coo_merge_runs. */
SKM_API size_t skm_learn_wide_workspace(int64_t nres);
SKM_API int skm_learn_wide(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                   const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t n_ann,
                   const uint64_t *d_sorted_codes, const int32_t *d_col_of_sorted, int64_t K,
                   uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_nnz, void *workspace,
                   size_t workspace_bytes, skm_stream_t stream);

/* ---- code spaces too large for tables (nsym^k > 2^27, up to 2^64 - 1: the alphabet/k sweep) ----------
 * (a7) basis of one shard as a table sorted by code: distinct window codes, their occurrence counts and the
 * position (res_base + index of the window's last residue) of their first occurrence — the dict of
 * kmerize.smk:89-104 before filtering and ordering.  Outputs need capacity nres; *d_n_out = entries.
 * One call handles < 2^30 residues. */
SKM_API size_t skm_basis_sorted_local_workspace(int64_t nres);
SKM_API int skm_basis_sorted_local(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets,
                           int64_t nseq, const uint8_t *d_lut, int nsym, int k, int64_t res_base,
                           uint64_t *d_codes_out, int64_t *d_counts_out, int64_t *d_first_out,
                           int64_t *d_n_out, void *workspace, size_t workspace_bytes,
                           skm_stream_t stream);
/* (a7) n table entries (the concatenated tables of chunks / GPUs; merged != 0: a single table, already
 * distinct and sorted) -> the basis: entries with equal codes are combined (sum of counts, min of first),
 * count > min_filter kept (kmerize.smk:97-104), ordered by first position.  d_basis_out / d_basis_counts_out
 * (nullable): codes and counts in first-occurrence order; d_sorted_codes_out + d_col_of_sorted_out: the kept
 * codes in ascending order with the basis column of each (the lookup structure of skm_count_csr_wide /
 * skm_codes_to_columns).  first_bound: an exclusive upper bound of the first positions (the total residue count
 * of all shards; <= 0 = unknown) — it limits the bits of the ordering sort.  All outputs need capacity n;
 * *d_K_out = basis size. */
SKM_API size_t skm_basis_sorted_finalize_workspace(int64_t n);
SKM_API int skm_basis_sorted_finalize(const uint64_t *d_codes, const int64_t *d_counts, const int64_t *d_first,
                              int64_t n, int merged, int64_t min_filter, int64_t first_bound,
                              uint64_t *d_basis_out,
                              int64_t *d_basis_counts_out, uint64_t *d_sorted_codes_out,
                              int32_t *d_col_of_sorted_out, int64_t *d_K_out, void *workspace,
                              size_t workspace_bytes, skm_stream_t stream);
/* basis column of each code (binary search in the sorted code list), -1 when the basis does not hold it:
 * the membership test of kmerize.smk:112-120 / the dict lookup of learn.smk:377-382 for 64-bit codes. */
SKM_API int skm_codes_to_columns(const uint64_t *d_codes, int64_t n, const uint64_t *d_sorted_codes,
                         const int32_t *d_col_of_sorted, int64_t K, int32_t *d_cols_out,
                         skm_stream_t stream);
/* (a11 at any nsym^k <= 2^64 - 1) per-sequence distinct window codes and their counts as CSR; a row's entries are
 * ordered by code.  With a basis (d_sorted_codes, d_col_of_sorted, K) entries outside it are dropped and
 * d_cols_out (nullable) receives the basis column of every entry; d_codes_out is nullable when d_cols_out is
 * given.  d_rowptr int64 [nseq+1]; entry outputs need capacity nres.  One call handles < 2^30 residues. */
SKM_API size_t skm_count_csr_wide_workspace(int64_t nres, int64_t nseq);
SKM_API int skm_count_csr_wide(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                       const uint8_t *d_lut, int nsym, int k, const uint64_t *d_sorted_codes,
                       const int32_t *d_col_of_sorted, int64_t K, int64_t *d_rowptr,
                       uint64_t *d_codes_out, uint32_t *d_cols_out, int32_t *d_vals, void *workspace,
                       size_t workspace_bytes, skm_stream_t stream);

/* Column sums of a COO matrix: d_totals[key % S] += value (d_totals int64 [S], accumulated, not cleared): the annotated
 * share of the Totals row (learn.smk:380) from the already aggregated matrix, one atomic per entry. */
SKM_API int skm_coo_colsum(const uint64_t *d_keys, const int64_t *d_vals, int64_t nnz, int64_t S,
                   int64_t *d_totals, skm_stream_t stream);

/* The same fan-in when the input is a concatenation of n_runs SORTED runs (what a rank receives from the all_to_all of
 * the sparse learn exchange): pairwise merge tree + reduce-by-key, ceil(log2 n_runs) + 1 streaming passes instead of a
 * radix sort.  run_offsets_host: HOST array [n_runs + 1] of entry offsets into d_keys_in / d_vals_in. */
SKM_API size_t skm_coo_merge_runs_workspace(int64_t n, int n_runs);
SKM_API int skm_coo_merge_runs(const uint64_t *d_keys_in, const int64_t *d_vals_in, const int64_t *run_offsets_host,
                       int n_runs, uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_n_out,
                       void *workspace, size_t workspace_bytes, skm_stream_t stream);

/* Annotation-major COO (key = ann * S + code) -> k-mer-major CSC for the SpMM:
 * d_colptr int64 [S+1], d_rows int32 [nnz] (annotation), d_mvals int32 [nnz] = M[a, c],
 * d_mnorm2 (nullable) = ||m_a||^2 (exact integer sum, as float64), d_inv_m32 (nullable) =
 * float32 1 / ||m_a|| (0 for empty rows), *d_max_m = largest entry (callers must check it
 * is < 2^31: larger entries do not fit d_mvals).  S <= 2^31 - 1 (S is the key stride: nsym^k, or the basis
 * column count of a matrix keyed by column). */
SKM_API size_t skm_csc_build_workspace(int64_t nnz, int64_t n_ann);
/* skm_csc_build_workspace for S columns: S may be up to 2^31 - 1 (a learned matrix keyed by basis column,
 * skm_learn_wide); for S <= SKM_DENSE_MAX_SPACE it equals skm_csc_build_workspace, which sizes for those. */
SKM_API size_t skm_csc_build_workspace_cols(int64_t nnz, int64_t n_ann, int64_t S);
SKM_API int skm_csc_build(const uint64_t *d_keys, const int64_t *d_vals, int64_t nnz, int64_t S,
                  int64_t n_ann, int64_t *d_colptr, int32_t *d_rows, int32_t *d_mvals,
                  double *d_mnorm2, float *d_inv_m32, int64_t *d_max_m, void *workspace,
                  size_t workspace_bytes, skm_stream_t stream);

/* (a16/a17 at large K) apply as SpMM: queries are CSR rows over CODES (skm_count_csr with
 * d_col_of_code = NULL, so that ||q|| runs over all valid k-mers, apply.smk:268-276).
 * Dots are accumulated EXACTLY in integer shared-memory accumulators (acc_bits = 32 when
 * max(M) * (largest row total of the queries) < 2^32, else 64); scores are
 * dot * (1/||q||) * (1/||m||) in float64 like skm_apply_dense, ties -> lowest index.
 * n_ann <= 51200 (32-bit) or 25600 (64-bit) per call: shard the annotations and merge with
 * skm_top2_merge.  d_qnorm2 (nullable) receives ||q||^2.  d_inv_m32 must be 16-byte aligned.
 * d_packed (nullable): the CSC entries as one 32-bit word each, value << 16 | annotation (skm_csc_pack; needs
 * n_ann <= 65536 and every value < 65536) — the kernel then reads half the bytes and pipelines its loads;
 * d_rows / d_mvals are not read in that case. */
SKM_API int skm_csc_pack(const int32_t *d_rows, const int32_t *d_mvals, int64_t nnz, uint32_t *d_packed,
                 skm_stream_t stream);
SKM_API int skm_apply_sparse(const int64_t *d_rowptr, const uint32_t *d_cols, const int32_t *d_vals,
                     int64_t nq, const int64_t *d_colptr, const int32_t *d_rows,
                     const int32_t *d_mvals, const uint32_t *d_packed, const double *d_mnorm2,
                     const float *d_inv_m32, int64_t n_ann, int acc_bits, int32_t *d_top1, int32_t *d_top2,
                     double *d_score1, double *d_score2, double *d_qnorm2,
                     skm_stream_t stream);
/* skm_apply_sparse that also writes every query's full cosine row, the association matrix of
 * apply.smk:282-299 (save_apply_associations) and learn.smk:821-849 (seq-annotation-scores-*.csv):
 * d_out_rows[q * ld_rows + a] for every q < nq and a < n_ann (float64, ld_rows >= n_ann, d_out_rows
 * non-NULL), each the exact score of skm_apply_sparse — exactly 0.0 when the integer dot is 0, so the
 * entries at d_top1 / d_top2 are bit-equal to d_score1 / d_score2.  Top-2 outputs as skm_apply_sparse,
 * bit for bit.  The rows are written with streaming stores; [q, a0, a0 + n_ann) slices of a wider
 * row-major buffer are what an annotation-sharded caller passes (d_out_rows offset by a0). */
SKM_API int skm_apply_sparse_rows(const int64_t *d_rowptr, const uint32_t *d_cols, const int32_t *d_vals,
                     int64_t nq, const int64_t *d_colptr, const int32_t *d_rows,
                     const int32_t *d_mvals, const uint32_t *d_packed, const double *d_mnorm2,
                     const float *d_inv_m32, int64_t n_ann, int acc_bits, int32_t *d_top1, int32_t *d_top2,
                     double *d_score1, double *d_score2, double *d_qnorm2, double *d_out_rows,
                     int64_t ld_rows, skm_stream_t stream);

/* (a16/a17) apply: cosine_similarity + top-2, apply.smk:278-335 and
 * learn.smk:811-849.  Queries are int32 count rows [nq, K] over the same
 * columns as d_M (int64 [n_ann, K]); d_qnorm2 holds ||q||^2 over ALL valid
 * query k-mers (the union re-index of apply.smk:268-276), d_mnorm2 ||m||^2.
 * Outputs per query: top-1 / top-2 annotation index (ties: lowest index) and
 * cosine in float64.  Dot products are exact integers (see DESIGN.md). */
SKM_API size_t skm_apply_dense_workspace(int64_t nq, int64_t n_ann, int64_t K);
SKM_API int skm_apply_dense(const int32_t *d_Q, int64_t nq, int64_t K,
                    const int64_t *d_M, int64_t n_ann, const double *d_qnorm2,
                    const double *d_mnorm2, int32_t *d_top1, int32_t *d_top2,
                    double *d_score1, double *d_score2, double *d_scores_full,
                    void *workspace, size_t workspace_bytes,
                    skm_stream_t stream);

/* (a16/a17) apply on the tensor cores (tcgen05.mma kind::i8, TMA-fed, TMEM accumulators) for
 * dense bases with K <= 32768.  The integer GEMM is exact: query counts must fit 8 bits and
 * the annotation matrix is split into n_planes <= 4 base-256 digit planes by
 * skm_apply_tc_prepare (once per learned matrix; this call synchronises the stream to read
 * back the largest entry).  d_planes needs skm_apply_tc_planes_bytes() bytes, 128-byte
 * aligned.  skm_apply_tc writes *d_status = 1 (device int) when a query count exceeded 255:
 * the outputs of THOSE rows are invalid and the caller re-scores them with skm_apply_dense
 * (skm_rows_out_of_range_i32 lists them); all other rows are exact.  Scores are
 * dot * (1/||q||) * (1/||m||) in float64; outputs as skm_apply_dense. */
SKM_API size_t skm_apply_tc_planes_bytes(int64_t n_ann, int64_t K);
SKM_API int skm_apply_tc_prepare(const int64_t *d_M, int64_t n_ann, int64_t K, uint8_t *d_planes,
                         size_t planes_bytes, int *n_planes_out, skm_stream_t stream);
SKM_API size_t skm_apply_tc_workspace(int64_t nq, int64_t K, int64_t n_ann);
SKM_API int skm_apply_tc(const int32_t *d_Q, int64_t nq, int64_t K, const uint8_t *d_planes,
                 int n_planes, int64_t n_ann, const double *d_qnorm2,
                 const double *d_mnorm2, int32_t *d_top1, int32_t *d_top2,
                 double *d_score1, double *d_score2, double *d_scores_full,
                 int *d_status, void *workspace, size_t workspace_bytes,
                 skm_stream_t stream);

/* Annotation-sharded apply (multi-GPU fan-in of apply.smk:312-335): merge per-shard top-2
 * lists into the global top-2.  d_idx is int64 [n_shards, 2, nq] with GLOBAL annotation
 * indices (-1 = no candidate), d_score float64 of the same shape.  Ties -> lowest index. */
SKM_API int skm_top2_merge(const int64_t *d_idx, const double *d_score, int64_t n_shards,
                   int64_t nq, int32_t *d_top1, int32_t *d_top2, double *d_score1,
                   double *d_score2, skm_stream_t stream);

/* row squared norms of an integer matrix (sklearn normalize, float64). */
SKM_API int skm_row_norm2_i32(const int32_t *d_X, int64_t rows, int64_t cols,
                      double *d_out, skm_stream_t stream);
SKM_API int skm_row_norm2_i64(const int64_t *d_X, int64_t rows, int64_t cols,
                      double *d_out, skm_stream_t stream);

/* KmerBasis.transform / KmerVec.harmonize, vectorize.py:54-119,330-345: column gather with
 * zero fill.  out[r, j] = in[r, idx[j]] (row-major [rows, n] -> [rows, p]); idx[j] outside
 * [0, n) gives a zero column.  elem_bytes in {1, 2, 4, 8}. */
SKM_API int skm_gather_columns(const void *d_in, int64_t rows, int64_t n, int elem_bytes,
                       const int64_t *d_idx, int64_t p, void *d_out,
                       skm_stream_t stream);

/* Merge.merge_dataframes / merge_with_base, learn.smk:467-494,556-579: outer join of count
 * matrices on their k-mer columns and row-wise sum.  dst[row_map[r], col_map[c]] +=
 * src[r, c] for int64 matrices; negative map entries drop the row / column. */
SKM_API int skm_scatter_add_i64(const int64_t *d_src, int64_t rows, int64_t cols,
                        const int64_t *d_row_map, const int64_t *d_col_map,
                        int64_t *d_dst, int64_t dst_rows, int64_t dst_cols,
                        skm_stream_t stream);

/* Compact transports of a dense count matrix [rows, cols] (in_bits 32 = int32, 16 = uint16) for the trip back to the
 * host — the reference's own vectorize payload is the 0/1 presence matrix (kmerize.smk:112-120,132-139).
 * skm_pack_counts_u8: uint8 counts; entries >= 255 are written as 255 and appended (unordered) to the escape list
 * (row, col, count), *d_n_esc (device int64) = how many there are (may exceed esc_capacity: the list is then
 * truncated and the caller must retry with a larger one).  Lossless: out[r, c] < 255 is the count itself.
 * skm_pack_presence_bits: bit (c & 7) of byte c >> 3 of a row of ceil(cols / 8) bytes is counts[r, c] > 0. */
SKM_API int skm_pack_counts_u8(const void *d_counts, int64_t rows, int64_t cols, int in_bits, uint8_t *d_out,
                       int32_t *d_esc_row, int32_t *d_esc_col, int32_t *d_esc_val, int64_t esc_capacity,
                       int64_t *d_n_esc, skm_stream_t stream);
SKM_API int skm_pack_presence_bits(const void *d_counts, int64_t rows, int64_t cols, int in_bits, uint8_t *d_out,
                           skm_stream_t stream);

/* Rows of an int32 matrix holding an element outside [lo, hi], appended (unordered) to d_rows_out; *d_n_out
 * (device int64) = how many.  skm_apply_tc scores rows with counts in 0..255; the caller re-scores the listed
 * rows with skm_apply_dense (apply.smk:278-289 has no such limit). */
SKM_API int skm_rows_out_of_range_i32(const int32_t *d_X, int64_t rows, int64_t cols, int32_t lo, int32_t hi,
                              int32_t *d_rows_out, int64_t capacity, int64_t *d_n_out, skm_stream_t stream);

/* Packed exchange format of a sorted COO list for the multi-GPU fan-in (Merge.merge_dataframes across ranks,
 * learn.smk:467-494): word = key << count_bits | count — 8 instead of 16 bytes per entry through the all_to_all and
 * the merge tree; words sort like keys.  skm_coo_pack sets *d_overflow (device int) when a count needs more than
 * count_bits or a key more than 64 - count_bits bits (the caller then uses the unpacked path).
 * skm_coo_merge_runs_packed: skm_coo_merge_runs for runs of packed words -> unpacked (keys, summed counts). */
SKM_API int skm_coo_pack(const uint64_t *d_keys, const int64_t *d_vals, int64_t n, int count_bits, uint64_t *d_packed,
                 int *d_overflow, skm_stream_t stream);
SKM_API size_t skm_coo_merge_runs_packed_workspace(int64_t n, int n_runs);
SKM_API int skm_coo_merge_runs_packed(const uint64_t *d_packed_in, const int64_t *run_offsets_host, int n_runs,
                              int count_bits, uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_n_out,
                              void *workspace, size_t workspace_bytes, skm_stream_t stream);

/* Multi-GPU fan-in over NVLink peer memory (one process per GPU; Merge.merge_dataframes across ranks, learn.smk:467-494).
 * The ONE exception to "the library never allocates": CUDA IPC exports whole allocations, so receive buffers are
 * cudaMalloc'ed here.  skm_peer_alloc returns the buffer and its 64-byte IPC handle (send it to the peers through the
 * host-side process group); skm_peer_open maps a peer's buffer into this process (enables peer access lazily);
 * skm_peer_close / skm_peer_free undo them.  These four calls synchronise like cudaMalloc / cudaFree.
 * skm_coo_pack_push: fused pack + all_to_all.  Entries [cut[r], cut[r+1]) of the local SORTED list (cut_host has world+1
 * values) are packed (skm_coo_pack's word format) and stored directly into rank r's receive buffer at entry offset
 * dst_off_host[r] (peer_bufs_host[r]; the own buffer for r == this rank).  The caller orders the step across ranks: a
 * collective before the call (nobody still reads its buffer) and one after it (all stores have landed). */
#define SKM_PEER_HANDLE_BYTES 64
SKM_API int skm_peer_alloc(size_t bytes, void **d_ptr, void *handle_out);
SKM_API int skm_peer_open(const void *handle, void **d_ptr);
SKM_API int skm_peer_close(void *d_ptr);
SKM_API int skm_peer_free(void *d_ptr);
SKM_API int skm_coo_pack_push(const uint64_t *d_keys, const int64_t *d_vals, const int64_t *cut_host, int world, int count_bits,
                      void *const *peer_bufs_host, const int64_t *dst_off_host, int *d_overflow, skm_stream_t stream);

/* (a12) learn for the heavy annotations: dense count rows (learn.smk:306-326,385-408 when a few families own most of
 * the sequences).  d_rows is uint32 [n_rows, S] (S = nsym^k <= 2^27), zeroed by the caller.
 * skm_rows_accumulate: rows[row_of_seq[s]][code] += 1 for every valid window of sequence s; sequences with
 *   row_of_seq < 0 are skipped.  Fast when the sequences of a row are adjacent (skm_gather_sequences): the row then
 *   stays in L2.  Fewer than 2^32 residues per call.
 * skm_rows_block_counts: d_counts int32 [n_rows, ceil(S / skm_rows_block())] = non-zeros per block of codes.
 * skm_rows_emit: the non-zeros of block (r, b), in code order, as (ann_of_row[r] * S + code, count) from
 *   d_keys_out[d_row_dst[r] + d_block_offsets[r * nblk + b]] on — the caller's exclusive prefix sums of the block
 *   counts inside a row and the place of the row's annotation in the merged sorted list.
 * skm_rows_colsum: d_totals[c] += sum over rows (the Totals row of learn.smk:380; not atomic: one launch at a time). */
SKM_API int skm_rows_accumulate(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                        const uint8_t *d_lut, int nsym, int k, const int32_t *d_row_of_seq, int64_t S,
                        uint32_t *d_rows, skm_stream_t stream);
SKM_API int skm_rows_block(void);
SKM_API int skm_rows_block_counts(const uint32_t *d_rows, int64_t n_rows, int64_t S, int32_t *d_counts, skm_stream_t stream);
SKM_API int skm_rows_emit(const uint32_t *d_rows, int64_t n_rows, int64_t S, const int64_t *d_block_offsets,
                  const int64_t *d_row_dst, const int64_t *d_ann_of_row, uint64_t *d_keys_out, int64_t *d_vals_out,
                  int64_t out_capacity, skm_stream_t stream);
SKM_API int skm_rows_colsum(const uint32_t *d_rows, int64_t n_rows, int64_t S, int64_t *d_totals, skm_stream_t stream);

/* Measurement helper (not on the product path): a kernel of `blocks` x 256 threads, each running 16 independent
 * chains of `iters` fp32 FMAs; *flops_out (host) = the flops it executes.  Timed with CUDA events by
 * scripts/measure_peaks.py it gives the fp32-FMA peak the sparse scoring roofline is quoted against (SURVEY 8(d)).
 * d_out: float [blocks * 256] (never written in practice). */
SKM_API int skm_bench_fma_f32(int64_t iters, int blocks, float *d_out, double *flops_out, skm_stream_t stream);

/* (a11) per-sequence counts as CSR WITHOUT a device-wide sort: a warp scans one sequence, sorts its window keys in
 * shared memory (bitonic network) and run-length encodes them; longer sequences get a CTA.  Same results as
 * skm_count_csr (key_bits = 32: keys = codes, or basis columns when d_col_of_code [S] is given; rows sorted by key)
 * and skm_count_csr_wide (key_bits = 64: keys = codes; with d_sorted_codes / d_col_of_sorted / K entries outside
 * the basis are dropped and d_cols_out (nullable) receives their columns).  d_keys_out: uint32 / uint64 [nres]
 * (nullable when d_cols_out is given).  max_len = longest sequence (<= 0: unknown).  < 2^30 residues per call. */
SKM_API size_t skm_count_csr_sorted_workspace(int64_t nres, int64_t nseq, int64_t max_len, int key_bits);
SKM_API int skm_count_csr_sorted(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                         const uint8_t *d_lut, int nsym, int k, int key_bits, const int32_t *d_col_of_code,
                         int64_t S, const uint64_t *d_sorted_codes, const int32_t *d_col_of_sorted, int64_t K,
                         int64_t max_len, int64_t *d_rowptr, void *d_keys_out, uint32_t *d_cols_out,
                         int32_t *d_vals, void *workspace, size_t workspace_bytes, skm_stream_t stream);

/* ---- confidence evaluation (rule `evaluate`, class Evaluator, learn.smk:923-1348) ----------------------
 * Read-back of a score matrix (learn.smk:964-981): per row of d_scores float64 [nq, n_ann] with NaN holes,
 * the column of the maximum (NaN skipped, first maximum = idxmax) and the two largest values; rows without
 * values give -1 / NaN. */
SKM_API int skm_top2_rows_f64(const double *d_scores, int64_t nq, int64_t n_ann, int32_t *d_top1,
                      int32_t *d_top2, double *d_score1, double *d_score2, skm_stream_t stream);
/* Difference bin of every query, 100 * -(round(score2 - score1, 2)) in 0..100 (255 when it is undefined:
 * no prediction, NaN, outside the 101 values of learn.smk:1063), written to d_bin_out (nullable), and — when
 * d_class is given — the crosstabs of learn.smk:1052-1061: d_hist_true / d_hist_false int64 [n_ann, 101]
 * += 1 at (top1, bin) for rows of class 1 (Known, True) / 2 (Known, False); class 0 rows are skipped.
 * The histograms are accumulated (not cleared), so files and shards add up. */
SKM_API int skm_confidence_hist(const int32_t *d_top1, const double *d_score1, const double *d_score2,
                        const uint8_t *d_class, int64_t nq, int64_t n_ann, int64_t *d_hist_true,
                        int64_t *d_hist_false, uint8_t *d_bin_out, skm_stream_t stream);
/* The d_class input of skm_confidence_hist for the rows of eval_apply (learn.smk:712-732), decided as
 * learn.smk:997-1008 decides it on the row label, without building the labels.  Row q is labelled
 * name[truth[q]] + "_known_" + decimal(row_base + q), or `<accession>_unknown_<n>` when truth[q] < 0.
 * Name table: UTF-8 bytes d_names, offsets int64 [n_names + 1]; entries 0 .. A-1 are the matrix's annotations
 * (the indices of d_top1), the rest any further names truth refers to.  d_class uint8 [nq]: 0 when the label
 * contains "unknown", else 1 when top1 >= 0 and name[top1] is a byte substring of the label, else 2.  An
 * index outside [0, n_names) names nothing.  row_base >= 0, row_base + nq <= 2^63 - 1. */
SKM_API int skm_confidence_classify(const int32_t *d_top1, const int32_t *d_truth, int64_t nq, int64_t row_base,
                            const uint8_t *d_names, const int64_t *d_name_offsets, int64_t n_names,
                            uint8_t *d_class, skm_stream_t stream);

/* ---- FASTA ingest (host cores, no device work): Bio.SeqIO.parse(f, "fasta") as kmerize.smk:90-129 uses it ----
 * text = the (decompressed) file in host memory.  A record starts at a '>' in column 0; id = the title up to its
 * first whitespace; sequence = the record's lines, each right-stripped, joined, blanks and CR removed.
 * skm_fasta_scan sizes the outputs; skm_fasta_pack writes residues [nres] back to back, offsets int64 [nseq+1],
 * the id bytes back to back and id_offsets int64 [nseq+1].  threads <= 0: all hardware threads. */
SKM_API int skm_fasta_scan(const uint8_t *text, int64_t nbytes, int threads, int64_t *nseq_out,
                   int64_t *nres_out, int64_t *idbytes_out);
SKM_API int skm_fasta_pack(const uint8_t *text, int64_t nbytes, int threads, uint8_t *residues_out,
                   int64_t *offsets_out, uint8_t *ids_out, int64_t *id_offsets_out);

/* ---- CSV interchange files formatted on the device (skm_csv.cu) -----------------------------------------------
 * The text of the reference's seq-annotation-scores files (apply.smk:295-299, learn.smk:821-849: pyarrow.csv.write_csv
 * of float64 columns and the string index column) and kmer-counts files (learn.smk:328-357 pandas layout,
 * :583-594 pyarrow layout).  Two passes: *_measure writes d_row_offsets int64 [rows + 1] (0, then the running byte
 * count after each row); *_write puts row r at d_text + d_row_offsets[r] - d_row_offsets[0], so a call over rows
 * [r0, r1) can pass d_row_offsets + r0 of a measure over more rows.  Workspace of a measure call:
 * skm_csv_rows_workspace(rows).  Row labels: UTF-8 bytes d_labels, absolute offsets int64 [rows + 1]
 * (d_label_offsets + r0 for a sub-range).
 *
 * float64 cells as pyarrow prints them: the shortest decimal that round-trips (closest of the shortest, ties to
 * even), decimal notation when the value is d.ddd x 10^x with -6 <= x <= 9 (no trailing ".0"), else d[.ddd]e+x /
 * d[.ddd]e-x; "nan" for any NaN, "inf", "-inf", "-0"; at most 25 bytes.  skm_csv_f64_host: the same function on the
 * host (out >= 25 bytes, no terminator), returns the length. */
SKM_API int skm_csv_f64_host(double v, char *out);
SKM_API size_t skm_csv_rows_workspace(int64_t rows);
/* Association rows: cells d_scores[r * ld + j] (j < A), each followed by ',', then the label in '"' with inner '"'
 * doubled, then '\n'. */
SKM_API int skm_csv_assoc_measure(const double *d_scores, int64_t rows, int64_t A, int64_t ld, const uint8_t *d_labels,
                          const int64_t *d_label_offsets, int64_t *d_row_offsets, void *workspace, size_t workspace_bytes,
                          skm_stream_t stream);
SKM_API int skm_csv_assoc_write(const double *d_scores, int64_t rows, int64_t A, int64_t ld, const uint8_t *d_labels,
                        const int64_t *d_label_offsets, const int64_t *d_row_offsets, uint8_t *d_text, skm_stream_t stream);
/* The top-2-masked association rows of eval_apply without save_associations (learn.smk:831-849): cell j of row r is
 * d_score2[r] when j == d_top2[r], else d_score1[r] when j == d_top1[r], else NaN ("nan"); no [rows, A] block. */
SKM_API int skm_csv_top2_measure(const int32_t *d_top1, const int32_t *d_top2, const double *d_score1, const double *d_score2,
                         int64_t rows, int64_t A, const uint8_t *d_labels, const int64_t *d_label_offsets,
                         int64_t *d_row_offsets, void *workspace, size_t workspace_bytes, skm_stream_t stream);
SKM_API int skm_csv_top2_write(const int32_t *d_top1, const int32_t *d_top2, const double *d_score1, const double *d_score2,
                       int64_t rows, int64_t A, const uint8_t *d_labels, const int64_t *d_label_offsets,
                       const int64_t *d_row_offsets, uint8_t *d_text, skm_stream_t stream);
/* Count rows from CSR over the file's K k-mer columns (d_rowptr int64 [rows + 1] absolute, d_cols int32 strictly
 * ascending in [0, K) within a row, d_vals int64; zero values count as absent) with the Sequence count / Kmer Count
 * fields d_seq_count / d_kmer_count int64 [rows].  layout 0 (learn.smk:328-357): label bytes verbatim (the caller
 * escapes them), then the two fields and the K cells, zeros blank.  layout 1 (learn.smk:583-594): the two fields and
 * the K cells with zeros as "0", then the label in '"' with inner '"' doubled.  Cells joined by ',', rows end in '\n'. */
SKM_API int skm_csv_counts_measure(const int64_t *d_rowptr, const int64_t *d_vals, int64_t rows, int64_t K,
                           const int64_t *d_seq_count, const int64_t *d_kmer_count, const uint8_t *d_labels,
                           const int64_t *d_label_offsets, int layout, int64_t *d_row_offsets, void *workspace,
                           size_t workspace_bytes, skm_stream_t stream);
SKM_API int skm_csv_counts_write(const int64_t *d_rowptr, const int32_t *d_cols, const int64_t *d_vals, int64_t rows, int64_t K,
                         const int64_t *d_seq_count, const int64_t *d_kmer_count, const uint8_t *d_labels,
                         const int64_t *d_label_offsets, int layout, const int64_t *d_row_offsets, uint8_t *d_text,
                         skm_stream_t stream);

/* Count-CSV parser (either layout; learn.smk:496-579 reads these files).  skm_csv_parse_rows: d_parity uint8 [nbytes]
 * = inclusive XOR scan of the '"' bytes (1 inside quotes); d_row_ends int64 [nbytes] receives the positions of the
 * '\n' bytes outside quotes in order, *d_nrows (device) their number.  Workspace: skm_csv_parse_workspace(nbytes).
 * skm_csv_parse_cells: row r is [d_row_start[r], d_row_end[r]] (its '\n' included), split into fields at ',' outside
 * quotes; d_role int32 [nfields] names each field: -1 the label (its byte range [d_label_start, d_label_end) is
 * written, quotes included), -2 Sequence count, -3 Kmer Count, j >= 0 k-mer column j.  A cell is empty (0), [0-9]+,
 * [0-9]+\.0* or d[.ddd]e[+-]x of an integer below 2^63.  With d_entry_offsets NULL: the count pass (d_row_nnz, the
 * two fields, the label ranges); else the write pass: the nonzero cells of row r as (d_cols, d_vals) from
 * d_entry_offsets[r], in column order.  *d_error (set to ~0 by the caller) takes the least (row << 32 | field) of a
 * malformed cell, field 0xFFFFFFFF for a row with a field count other than nfields.  rows < 2^31. */
SKM_API size_t skm_csv_parse_workspace(int64_t nbytes);
SKM_API int skm_csv_parse_rows(const uint8_t *d_text, int64_t nbytes, uint8_t *d_parity, int64_t *d_row_ends, int64_t *d_nrows,
                       void *workspace, size_t workspace_bytes, skm_stream_t stream);
SKM_API int skm_csv_parse_cells(const uint8_t *d_text, const uint8_t *d_parity, const int64_t *d_row_start,
                        const int64_t *d_row_end, int64_t rows, const int32_t *d_role, int nfields,
                        const int64_t *d_entry_offsets, int64_t *d_row_nnz, int64_t *d_seq_count, int64_t *d_kmer_count,
                        int64_t *d_label_start, int64_t *d_label_end, int32_t *d_cols, int64_t *d_vals,
                        unsigned long long *d_error, skm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SKM_B200_H */
