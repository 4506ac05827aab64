// skm_sparse.cu — sort-based (atomic-free) sparse paths for large k-mer bases.
//
//  skm_learn_sparse   kernel (c) for bases that do not fit a shared-memory row
//                     (learn.smk:306-326,359-408 at K ~ 1e6): every valid window of an
//                     annotated sequence becomes the 64-bit key  ann * S + code;  the keys of a
//                     shard are radix-sorted and run-length encoded into a sorted COO
//                     (key, count) list = the annotation x k-mer count matrix.  No atomics,
//                     bit-reproducible.  Unannotated sequences only feed the Totals table
//                     (skm_basis_accumulate gives it).
//  skm_learn_wide     the same list over code spaces beyond the tables (up to 2^64 - 1), keyed by BASIS COLUMN:
//                     ann * K + col, with a rest row for the unannotated sequences whose column sums are the Totals.
//  skm_coo_merge      sum of COO lists with equal keys (sort by key + reduce by key):
//                     Merge.merge_dataframes (learn.smk:467-494) for sparse matrices, and the
//                     fan-in after an all-gather of per-GPU lists.
//  skm_csc_build      annotation-major COO -> k-mer-major CSC (annotation index + int32 count per
//                     entry), exact ||m_a||^2 and float32 1 / ||m_a|| for the screening pass.
//  skm_apply_sparse   kernel (d) as SpMM with EXACT integer dots: one CTA per query keeps one
//                     integer accumulator per annotation in shared memory (up to 51,200), its
//                     warps walk the CSC columns of the query's k-mers and add count x M[a, c]
//                     with shared-memory integer atomics (order-independent, hence reproducible),
//                     then scan the accumulators for the top-2 (float32 screening, exact float64
//                     scores for the survivors; apply.smk:278-335).
//  skm_apply_sparse_rows  the same kernel that also streams every query's full cosine row out of the scan (the
//                     association matrix, apply.smk:295-299 / learn.smk:821-849).
//  window_keys_kernel is also the key generator of skm_count_csr (skm_count.cu).
#include <vector>

#include <cub/cub.cuh>

#include "skm_common.cuh"
#include "skm_tile.cuh"

namespace skm {

constexpr int SP_SEG = ts_seg_cap(28);                     // 7168 positions per staged segment
constexpr int SP_SYM_BYTES = (ts_sym_bytes(SP_SEG) + 15) & ~15;
template <typename KeyT> constexpr int sp_smem_bytes() { return SP_SYM_BYTES + SP_SEG * int(sizeof(KeyT)); }   // symbols + staged keys

// keys[p] for every residue position p of [off[0], off[nseq]) (p = position of the window's LAST residue):
//   MODE 0: column (col_of_code) or code, 32-bit, all-ones when invalid / filtered
//   MODE 1: (ann_id[row] - ann_lo) * S + code, `invalid` (one past the largest key, or all-ones) when the window is
//           invalid or the sequence's annotation is outside [ann_lo, ann_hi): the sort then only needs the bits of
//           the largest key.  32-bit keys when (ann_hi - ann_lo) * S < 2^32 (skm_learn_sparse_group).
template <int MODE, typename KeyT>
__global__ void __launch_bounds__(TS_THREADS) window_keys_kernel(const uint8_t *__restrict__ res, int64_t nres,
                                                                 const int64_t *__restrict__ off, int64_t nseq,
                                                                 const uint8_t *__restrict__ lut, uint32_t nsym, int k,
                                                                 uint32_t pow_k1, const int32_t *__restrict__ col_of_code,
                                                                 const int32_t *__restrict__ ann_id, uint64_t S,
                                                                 KeyT invalid, KeyT *__restrict__ keys, int32_t ann_lo = 0,
                                                                 int32_t ann_hi = 0x7FFFFFFF) {
    extern __shared__ __align__(128) uint8_t s_sym[];
    __shared__ uint8_t s_lut[256];
    __shared__ int64_t s_ctl[4];
    KeyT *s_keys = reinterpret_cast<KeyT *>(s_sym + SP_SYM_BYTES);       // one key per position of the staged segment
    ts_lut_init(s_lut, lut);
    __syncthreads();
    int64_t ann_row = -2;          // row whose annotation is cached
    uint64_t ann_base = ~0ull;
    ts_range_scan_rows<uint32_t>(res, nres, off, nseq, s_lut, s_sym, SP_SEG, k, nsym, pow_k1, /*origin=*/0, s_ctl,
                                 [&](int64_t, int64_t row, uint32_t code, bool ok, int local) {
                                     KeyT key = invalid;
                                     if (ok) {
                                         if (MODE == 0) {
                                             if (col_of_code) { const int32_t c = __ldg(col_of_code + code); if (c >= 0) key = KeyT(c); }
                                             else key = KeyT(code);
                                         } else {
                                             if (row != ann_row) {
                                                 ann_row = row;
                                                 const int32_t a = __ldg(ann_id + row);
                                                 ann_base = (a >= ann_lo && a < ann_hi) ? uint64_t(a - ann_lo) * S : ~0ull;
                                             }
                                             if (ann_base != ~0ull) key = KeyT(ann_base + code);
                                         }
                                     }
                                     s_keys[local] = key;
                                 },
                                 [&](int64_t rel_a, int n) {         // coalesced copy of the segment's keys
                                     for (int i = threadIdx.x; i < n; i += blockDim.x) keys[rel_a + i] = s_keys[i];
                                 });
}

// keys[p] for the wide learn (skm_learn_wide): a * K + col for the window whose last residue sits at p, with col its
// basis column (bucketed binary search) and a = ann_id[row], or n_ann (the rest row) when the sequence has no annotation
// in [0, n_ann); `invalid` when the window is invalid or its code is not in the basis
__global__ void __launch_bounds__(TS_THREADS) learn_wide_keys_kernel(const uint8_t *__restrict__ res, int64_t nres,
                                                                     const int64_t *__restrict__ off, int64_t nseq,
                                                                     const uint8_t *__restrict__ lut, uint64_t nsym, int k,
                                                                     uint64_t pow_k1, const int32_t *__restrict__ ann_id,
                                                                     int64_t n_ann, SortedBasis sb, uint64_t invalid,
                                                                     uint64_t *__restrict__ keys) {
    extern __shared__ __align__(128) uint8_t s_sym[];
    __shared__ uint8_t s_lut[256];
    __shared__ int64_t s_ctl[4];
    uint64_t *s_keys = reinterpret_cast<uint64_t *>(s_sym + SP_SYM_BYTES);
    ts_lut_init(s_lut, lut);
    __syncthreads();
    int64_t ann_row = -2;          // row whose annotation is cached
    uint64_t ann_base = 0;
    ts_range_scan_rows<uint64_t>(res, nres, off, nseq, s_lut, s_sym, SP_SEG, k, nsym, pow_k1, /*origin=*/0, s_ctl,
                                 [&](int64_t, int64_t row, uint64_t code, bool ok, int local) {
                                     uint64_t key = invalid;
                                     if (ok) {
                                         const int32_t c = sorted_lookup(sb, code);
                                         if (c >= 0) {
                                             if (row != ann_row) {
                                                 ann_row = row;
                                                 const int32_t a = __ldg(ann_id + row);
                                                 ann_base = uint64_t(a >= 0 && a < n_ann ? int64_t(a) : n_ann) * uint64_t(sb.K);
                                             }
                                             key = ann_base + uint64_t(c);
                                         }
                                     }
                                     s_keys[local] = key;
                                 },
                                 [&](int64_t rel_a, int n) {         // coalesced copy of the segment's keys
                                     for (int i = threadIdx.x; i < n; i += blockDim.x) keys[rel_a + i] = s_keys[i];
                                 });
}

int wide_check(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut,
               int nsym, int k, const char *who, unsigned __int128 *S);      // skm_wide.cu

// the runs of the invalid key (and of the all-ones fill outside the sequences) sort last: drop them
__global__ void coo_finish_kernel(const uint64_t *__restrict__ uniq, const int64_t *__restrict__ num_runs, uint64_t invalid,
                                  int64_t *__restrict__ nnz) {
    int64_t n = *num_runs;
    while (n > 0 && uniq[n - 1] >= invalid) --n;
    *nnz = n;
}

// ---- CSC build -------------------------------------------------------------------------------
// ||m_a||^2 as exact integers (order-independent, hence reproducible).  Entries are < 2^31 (skm_csc_build's callers
// check max_m) and an annotation's entries sum to at most the residues it was learned from, so sum v^2 <= (sum v)^2
// stays below 2^64 while an annotation holds fewer than 2^32 k-mer occurrences; the dense kernel (row_norm2_kernel)
// accumulates in 128 bits and gives the same integer.
__global__ void __launch_bounds__(256) coo_row_norm2_kernel(const uint64_t *__restrict__ keys, const int64_t *__restrict__ vals,
                                                            int64_t nnz, uint64_t S, unsigned long long *__restrict__ norm2) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nnz; i += int64_t(gridDim.x) * blockDim.x) {
        const unsigned long long v = (unsigned long long)vals[i];
        atomicAdd(norm2 + keys[i] / S, v * v);
    }
}
__global__ void __launch_bounds__(256) csc_keys_kernel(const uint64_t *__restrict__ keys, int64_t nnz, uint64_t S,
                                                       uint64_t n_ann, uint64_t *__restrict__ out, int64_t *__restrict__ perm) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nnz; i += int64_t(gridDim.x) * blockDim.x) {
        const uint64_t a = keys[i] / S, c = keys[i] - a * S;
        out[i] = c * n_ann + a;
        perm[i] = i;
    }
}
__global__ void __launch_bounds__(256) csc_emit_kernel(const uint64_t *__restrict__ skeys, const int64_t *__restrict__ perm,
                                                       const int64_t *__restrict__ vals, int64_t nnz, uint64_t n_ann,
                                                       int32_t *__restrict__ rows, int32_t *__restrict__ mvals,
                                                       unsigned long long *__restrict__ colcount, unsigned long long *__restrict__ max_m) {
    unsigned long long mx = 0;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nnz; i += int64_t(gridDim.x) * blockDim.x) {
        const uint64_t c = skeys[i] / n_ann, a = skeys[i] - c * n_ann;
        rows[i] = int32_t(a);
        const unsigned long long v = (unsigned long long)vals[perm[i]];
        mvals[i] = int32_t(v);                 // callers check *max_m < 2^31
        mx = v > mx ? v : mx;
        atomicAdd(colcount + c + 1, 1ull);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long x = __shfl_xor_sync(FULL, mx, o); mx = x > mx ? x : mx; }
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(max_m, mx);
}
__global__ void norm2_finish_kernel(const unsigned long long *__restrict__ in, int64_t n, double *__restrict__ norm2, float *__restrict__ inv32) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        const double m2 = double(in[i]);
        if (norm2) norm2[i] = m2;
        if (inv32) inv32[i] = m2 > 0.0 ? float(1.0 / sqrt(m2)) : 0.0f;
    }
}

// ---- SpMM + top-2 ------------------------------------------------------------------------------
struct Top2d {
    double s1, s2;
    int i1, i2;
};
// higher score first; equal scores -> lower annotation index (np.argsort(-S) on exact ties)
__device__ __forceinline__ void top2d_push(Top2d &t, double s, int i) {
    if (i < 0) return;
    if (t.i1 < 0 || s > t.s1 || (s == t.s1 && i < t.i1)) { t.s2 = t.s1; t.i2 = t.i1; t.s1 = s; t.i1 = i; }
    else if (t.i2 < 0 || s > t.s2 || (s == t.s2 && i < t.i2)) { t.s2 = s; t.i2 = i; }
}
// Per-thread running top-2 of the accumulator scan, ordered by the float32 screening score dot / ||m|| whenever two
// scores differ by more than 1e-5 relative (their float32 error is < 4e-7); near-ties are settled by the exact
// float64 scores, tie -> lower index.  The same scheme as the tensor-core kernel (skm_apply_tc.cu).
struct Top2x {
    float f1, f2;
    unsigned long long d1, d2;      // exact dots
    int i1, i2;
};
__device__ __forceinline__ double sp_exact(unsigned long long dot, double inv_qn, const double *__restrict__ mnorm2, int a) {
    return double(dot) * (inv_qn * (1.0 / sqrt(mnorm2[a])));
}
__device__ __forceinline__ bool sp_above(float f, unsigned long long dot, int i, float fk, unsigned long long dk, int ik, double inv_qn,
                                         const double *__restrict__ mnorm2) {
    if (f > fk * 1.00001f) return true;
    if (f < fk * 0.99999f) return false;
    const double s = sp_exact(dot, inv_qn, mnorm2, i), sk = sp_exact(dk, inv_qn, mnorm2, ik);
    return s > sk || (s == sk && i < ik);
}
__device__ __forceinline__ void top2x_push(Top2x &t, float f, unsigned long long dot, int i, double inv_qn, const double *__restrict__ mnorm2) {
    if (t.i1 < 0 || sp_above(f, dot, i, t.f1, t.d1, t.i1, inv_qn, mnorm2)) {
        t.f2 = t.f1; t.d2 = t.d1; t.i2 = t.i1;
        t.f1 = f; t.d1 = dot; t.i1 = i;
    } else if (t.i2 < 0 || sp_above(f, dot, i, t.f2, t.d2, t.i2, inv_qn, mnorm2)) {
        t.f2 = f; t.d2 = dot; t.i2 = i;
    }
}

constexpr int SPA_THREADS = 512;
constexpr int SPA_EB = 512;        // query entries staged per block (one per thread: SPA_EB <= SPA_THREADS)
static_assert(SPA_EB <= SPA_THREADS, "the staging step gives every staged query entry its own thread");
constexpr int SPA_SEG = 512;       // CSC entries per segment (16 per lane)

// acc[w & 0xFFFF] += c * (w >> 16): one red.shared.add on the 32-bit shared address `acc` (address of accumulator 0),
// no predicate and no branch — a lane without an entry adds 0 to a dummy accumulator of its own behind the real ones.
// Annotation in the LOW half: the address is one mask + one scaled add, the value one shift (5 instructions per entry
// with the multiply and the red).
template <typename AccT> __device__ __forceinline__ void spa_red_add(uint32_t acc, uint32_t w, uint32_t c);
template <> __device__ __forceinline__ void spa_red_add<uint32_t>(uint32_t acc, uint32_t w, uint32_t c) {
    uint32_t a;
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(a) : "r"(w & 0xFFFFu), "r"(acc));       // one mask + one multiply-add
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(c * (w >> 16)) : "memory");
}
template <> __device__ __forceinline__ void spa_red_add<unsigned long long>(uint32_t acc, uint32_t w, uint32_t c) {
    uint32_t a;
    asm("mad.lo.u32 %0, %1, 8, %2;" : "=r"(a) : "r"(w & 0xFFFFu), "r"(acc));
    asm volatile("red.shared.add.u64 [%0], %1;" ::"r"(a), "l"((unsigned long long)c * (w >> 16)) : "memory");
}
constexpr int SPA_DUMMY = 32;      // dummy accumulators behind the padded real ones: one per lane

// One CTA per query (grid-stride).  acc: one integer per annotation in shared memory (AccT = uint32 when every dot
// fits 32 bits — the host checks max(M) * max row total < 2^32 — else uint64).
//   walk   the query's (k-mer, count) entries are staged in shared memory with their column ranges; the warps share
//          the columns segment by segment: acc[row] += count * M[row, code].
//   scan   every thread owns the same accumulators for every query (4 adjacent ones per step): float32 screening
//          score acc * inv_m32 against the thread's running runner-up, survivors inserted into a Top2x; the
//          accumulators are zeroed on the way.  The threads' top-2 lists are then merged with exact float64 scores.
// ROWS: the scan also writes rows_out[q * ld + a] for every a < n_ann — sp_exact's value, exactly 0.0 for a zero dot
// (which covers a zero-norm annotation and a query without a valid window) — so the row's entries at top1 / top2 are
// bit-equal to score1 / score2.  Streaming stores: the CSC is what should stay in L2.
template <typename AccT, bool PACKED, bool ROWS>
__global__ void __launch_bounds__(SPA_THREADS, 1)
apply_sparse_kernel(const int64_t *__restrict__ rowptr, const uint32_t *__restrict__ qcols, const int32_t *__restrict__ qvals,
                    int64_t nq, const int64_t *__restrict__ colptr, const int32_t *__restrict__ rows,
                    const int32_t *__restrict__ mvals, const uint32_t *__restrict__ packed,
                    const double *__restrict__ mnorm2, const float *__restrict__ inv_m32,
                    int n_ann, int32_t *__restrict__ top1, int32_t *__restrict__ top2, double *__restrict__ sc1,
                    double *__restrict__ sc2, double *__restrict__ qnorm2_out, double *__restrict__ rows_out, int64_t ld) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    __shared__ unsigned long long s_n2;
    __shared__ Top2d s_top[SPA_THREADS / 32];
    __shared__ int64_t s_p0[SPA_EB];
    __shared__ int s_len[SPA_EB];
    __shared__ uint32_t s_cnt[SPA_EB];
    __shared__ int s_first[SPA_EB + 1];                 // segments of the block's entries before entry j (exclusive prefix)
    __shared__ int s_wtot[SPA_THREADS / 32];
    AccT *acc = reinterpret_cast<AccT *>(s_raw);
    const uint32_t acc_addr = smem_addr(acc);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = SPA_THREADS / 32;
    constexpr int PER = 16 / sizeof(AccT);                 // accumulators per 16-byte step of the scan
    const int n_pad = (n_ann + PER - 1) / PER * PER;
    const uint32_t pad_word = uint32_t(n_pad + lane);                // packed path: (value 0, dummy accumulator of this lane)
    for (int i = tid; i < n_pad + SPA_DUMMY; i += SPA_THREADS) acc[i] = 0;
    if (tid == 0) s_n2 = 0;
    __syncthreads();
    for (int64_t q = blockIdx.x; q < nq; q += gridDim.x) {
        const int64_t e0 = __ldg(rowptr + q), e1 = __ldg(rowptr + q + 1);
        // ---- blocks of SPA_EB query entries are staged in shared memory; every column is cut into segments of SPA_SEG
        // entries, the (entry, segment) items are dealt round-robin to the warps, so that long columns (popular k-mers
        // meet thousands of annotations) spread over the CTA.  A lane loads its SPA_SEG / 32 entries of the segment
        // before the first atomic: the loads of a segment are all in flight together. ----
        unsigned long long n2 = 0;
        for (int64_t b0 = e0; b0 < e1; b0 += SPA_EB) {
            const int nb = (e1 - b0 < SPA_EB) ? int(e1 - b0) : SPA_EB;
            // stage entry tid (nb <= SPA_EB <= SPA_THREADS) and scan the entries' segment counts: the block's work is the
            // list of (entry, segment) items, item t = s_first[j] + s
            int nseg = 0;
            if (tid < nb) {
                const uint32_t c = __ldg(qcols + b0 + tid);
                const uint32_t cnt = uint32_t(__ldg(qvals + b0 + tid));
                const int64_t p0 = __ldg(colptr + c);
                const int len = int(__ldg(colptr + c + 1) - p0);
                s_p0[tid] = p0;
                s_len[tid] = len;
                s_cnt[tid] = cnt;
                n2 += (unsigned long long)cnt * cnt;
                nseg = (len + SPA_SEG - 1) / SPA_SEG;
            }
            int incl = nseg;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
            if (lane == 31) s_wtot[warp] = incl;
            __syncthreads();
            int before = 0;
            for (int w = 0; w < warp; ++w) before += s_wtot[w];
            if (tid < nb) s_first[tid] = before + incl - nseg;
            // the total: the LAST thread's inclusive prefix (with nb == SPA_EB == SPA_THREADS there is no thread `nb` that
            // could write it — round 1 left s_first[SPA_EB] stale for queries with 512 or more distinct k-mers in a block)
            if (tid == SPA_THREADS - 1) s_first[nb] = before + incl;
            __syncthreads();
            const int n_items = s_first[nb];
            // ---- walk: item t goes to warp t mod NW; a lane first finds (entry, segment) of one of its warp's next 32
            // items by binary search in s_first, then the warp processes them one after the other.  (The first version
            // let every warp loop over ALL entries and skip those without a segment for it: 85 % of 541 M loop trips did
            // nothing — 23 % of the kernel's samples — and the warps finished unevenly: 15 % barrier stalls.) ----
            for (int base = warp; base < n_items; base += 32 * NW) {
                const int t = base + lane * NW;
                int ej = 0, es = 0;
                if (t < n_items) {
                    int lo = 0, hi = nb;                            // last j with s_first[j] <= t
                    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_first[mid] <= t) lo = mid; else hi = mid; }
                    ej = lo;
                    es = t - s_first[lo];
                }
                const int in_round = min(32, (n_items - base + NW - 1) / NW);
                if (PACKED) {
                    // one 32-bit word per CSC entry (annotation << 16 | value): half the loads and registers, which pays
                    // for a software pipeline — the next item's 8 loads are issued before the current item's atomics
                    // (22 % of the samples of the unpacked kernel wait on the loads of the item they are about to use)
                    uint32_t b0[SPA_SEG / 32], b1[SPA_SEG / 32], b2[SPA_SEG / 32];
                    auto fetch = [&](int i, uint32_t (&dst)[SPA_SEG / 32]) -> uint32_t {
                        const int j = __shfl_sync(FULL, ej, i), seg = __shfl_sync(FULL, es, i);
                        const int64_t pb = s_p0[j] + int64_t(seg) * SPA_SEG;
                        const int n = min(SPA_SEG, s_len[j] - seg * SPA_SEG);
#pragma unroll
                        for (int u = 0; u < SPA_SEG / 32; ++u) { const int idx = lane + 32 * u; dst[u] = (idx < n) ? __ldg(packed + pb + idx) : pad_word; }
                        return s_cnt[j];
                    };
                    // acc[word & 0xFFFF] += count * (word >> 16) as ONE unpredicated red.shared on a 32-bit shared address; a
                    // lane without an entry holds pad_word = (its dummy accumulator, value 0).  The compiler's version of
                    // `if (w & 0xFFFF) atomicAdd(...)` was a branch with a reconvergence barrier around every atomic plus the
                    // recomputation of the shared window base: 11 instructions per entry instead of 5.
                    auto add_all = [&](const uint32_t (&w)[SPA_SEG / 32], uint32_t c) {
#pragma unroll
                        for (int u = 0; u < SPA_SEG / 32; ++u) spa_red_add<AccT>(acc_addr, w[u], c);
                    };
                    // two items of look-ahead (16 loads per lane in flight while the current item's atomics run); the three
                    // buffers rotate by name, not by register moves
                    uint32_t c0 = fetch(0, b0), c1 = 0, c2 = 0;
                    if (in_round > 1) c1 = fetch(1, b1);
                    for (int i = 0; i < in_round; i += 3) {
                        if (i + 2 < in_round) c2 = fetch(i + 2, b2);
                        add_all(b0, c0);
                        if (i + 1 >= in_round) break;
                        if (i + 3 < in_round) c0 = fetch(i + 3, b0);
                        add_all(b1, c1);
                        if (i + 2 >= in_round) break;
                        if (i + 4 < in_round) c1 = fetch(i + 4, b1);
                        add_all(b2, c2);
                    }
                    continue;
                }
                for (int i = 0; i < in_round; ++i) {
                    const int j = __shfl_sync(FULL, ej, i), seg = __shfl_sync(FULL, es, i);
                    const int len = s_len[j];
                    const AccT cnt = AccT(s_cnt[j]);
                    const int64_t pb = s_p0[j] + int64_t(seg) * SPA_SEG;
                    const int n = min(SPA_SEG, len - seg * SPA_SEG);
                    int r[SPA_SEG / 32];
                    uint32_t m[SPA_SEG / 32];
#pragma unroll
                    for (int u = 0; u < SPA_SEG / 32; ++u) {
                        const int idx = lane + 32 * u;
                        r[u] = -1;
                        m[u] = 0;
                        if (idx < n) { r[u] = __ldg(rows + pb + idx); m[u] = uint32_t(__ldg(mvals + pb + idx)); }
                    }
#pragma unroll
                    for (int u = 0; u < SPA_SEG / 32; ++u)
                        if (r[u] >= 0) atomicAdd(&acc[r[u]], cnt * AccT(m[u]));
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(FULL, n2, o);
        if (lane == 0 && n2) atomicAdd(&s_n2, n2);
        __syncthreads();
        // ---- scan ----
        const double qn2 = double(s_n2);
        const double inv_qn = qn2 > 0.0 ? 1.0 / sqrt(qn2) : 0.0;
        Top2x bx{0.f, 0.f, 0ull, 0ull, -1, -1};
        float thr = 1e-30f;                                    // > 0: zero dots are never candidates (see the final fill)
        for (int a0 = tid * PER; a0 < n_pad; a0 += SPA_THREADS * PER) {
            AccT v[PER];
            // the screening factors are loaded up front (one coalesced vector, independent of the accumulators): loaded
            // per non-zero accumulator they put an L2 round trip in front of every multiply
            float inv[PER];
            if (a0 + PER <= n_ann) {
                if (PER == 4) *reinterpret_cast<float4 *>(inv) = __ldg(reinterpret_cast<const float4 *>(inv_m32 + a0));
                else *reinterpret_cast<float2 *>(inv) = __ldg(reinterpret_cast<const float2 *>(inv_m32 + a0));
            } else {
#pragma unroll
                for (int i = 0; i < PER; ++i) inv[i] = (a0 + i < n_ann) ? __ldg(inv_m32 + a0 + i) : 0.f;
            }
            *reinterpret_cast<uint4 *>(v) = *reinterpret_cast<const uint4 *>(&acc[a0]);
            if constexpr (ROWS) {
                double *dst = rows_out + q * ld + a0;
#pragma unroll
                for (int i = 0; i < PER; ++i)
                    if (a0 + i < n_ann) __stcs(dst + i, v[i] != 0 ? sp_exact((unsigned long long)v[i], inv_qn, mnorm2, a0 + i) : 0.0);
            }
            bool any = false;
#pragma unroll
            for (int i = 0; i < PER; ++i) any |= (v[i] != 0);
            if (any) {
                *reinterpret_cast<uint4 *>(&acc[a0]) = make_uint4(0u, 0u, 0u, 0u);
                // group screening: ONE comparison of the group's largest float32 score against the threshold; the
                // per-accumulator path (insertion into the running top-2) runs only for a group that holds a candidate.
                // A zero dot gives 0 < thr, so zero dots are never candidates.  (One branchy copy of the insertion per
                // accumulator made the scan 25 % of the kernel's instructions.)
                float f[PER];
                float fm = 0.f;
#pragma unroll
                for (int i = 0; i < PER; ++i) { f[i] = float(v[i]) * inv[i]; fm = fmaxf(fm, f[i]); }
                if (fm >= thr) {
#pragma unroll
                    for (int i = 0; i < PER; ++i) {
                        if (f[i] >= thr) {
                            top2x_push(bx, f[i], (unsigned long long)v[i], a0 + i, inv_qn, mnorm2);
                            if (bx.i2 >= 0) thr = fmaxf(thr, bx.f2 * 0.99999f);
                        }
                    }
                }
            }
        }
        Top2d best{0.0, 0.0, -1, -1};
        if (bx.i1 >= 0) { best.i1 = bx.i1; best.s1 = sp_exact(bx.d1, inv_qn, mnorm2, bx.i1); }
        if (bx.i2 >= 0) { best.i2 = bx.i2; best.s2 = sp_exact(bx.d2, inv_qn, mnorm2, bx.i2); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double os1 = __shfl_xor_sync(FULL, best.s1, o), os2 = __shfl_xor_sync(FULL, best.s2, o);
            const int oi1 = __shfl_xor_sync(FULL, best.i1, o), oi2 = __shfl_xor_sync(FULL, best.i2, o);
            top2d_push(best, os1, oi1);
            top2d_push(best, os2, oi2);
        }
        if (lane == 0) s_top[warp] = best;
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < NW; ++w) { top2d_push(best, s_top[w].s1, s_top[w].i1); top2d_push(best, s_top[w].s2, s_top[w].i2); }
            // annotations that were never candidates score exactly 0: a missing winner / runner-up is the lowest-index one of them
            if (best.i1 < 0) { best.i1 = 0; best.s1 = 0.0; }
            if (best.i2 < 0 && n_ann > 1) { best.i2 = (best.i1 == 0) ? 1 : 0; best.s2 = 0.0; }
            top1[q] = best.i1; sc1[q] = best.s1;
            top2[q] = best.i2; sc2[q] = best.i2 >= 0 ? best.s2 : nan("");
            if (qnorm2_out) qnorm2_out[q] = qn2;
            s_n2 = 0;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) csc_pack_kernel(const int32_t *__restrict__ rows, const int32_t *__restrict__ mvals, int64_t nnz,
                                                       uint32_t *__restrict__ packed) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nnz; i += int64_t(gridDim.x) * blockDim.x)
        packed[i] = (uint32_t(mvals[i]) << 16) | (uint32_t(rows[i]) & 0xFFFFu);      // value high, annotation low
}


}  // namespace skm

extern "C" {

// window keys for skm_count_csr (declared in skm_count.cu)
int skm_window_keys_u32(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                        const uint8_t *d_lut, int nsym, int k, const int32_t *d_col_of_code, uint32_t *d_keys,
                        cudaStream_t st) {
    using namespace skm;
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    int64_t grid = int64_t(sm_count()) * 8;
    const int64_t max_grid = (nres + SP_SEG - 1) / SP_SEG;
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    window_keys_kernel<0, uint32_t><<<(unsigned)grid, TS_THREADS, sp_smem_bytes<uint32_t>(), st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k,
                                                                                      pow_k1, d_col_of_code, nullptr, 0, 0xFFFFFFFFu, d_keys);
    SKM_LAUNCH_CHECK("window_keys_kernel<0>");
    return SKM_OK;
}

size_t skm_learn_sparse_workspace(int64_t nres) {
    using namespace skm;
    if (nres <= 0) return 256;
    size_t t_sort = 0, t_rle = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, t_sort, (const uint64_t *)nullptr, (uint64_t *)nullptr, nres, 0, 64);
    cub::DeviceRunLengthEncode::Encode(nullptr, t_rle, (const uint64_t *)nullptr, (uint64_t *)nullptr, (int64_t *)nullptr,
                                       (int64_t *)nullptr, (int)std::min<int64_t>(nres, (1ll << 31) - 1));
    return 2 * align256(size_t(nres) * 8) + align256(std::max(t_sort, t_rle)) + 1024;
}

int skm_learn_sparse(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                     const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t n_ann,
                     uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_nnz, void *workspace,
                     size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    if (!ts_supported(nsym, k)) { set_error("skm_learn_sparse: nsym=%d k=%d outside the kernel envelope", nsym, k); return SKM_ERR_UNSUPPORTED; }
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (S128 >= ((unsigned __int128)1 << 32)) { set_error("skm_learn_sparse: code space must be < 2^32"); return SKM_ERR_UNSUPPORTED; }
    if (n_ann < 0 || (unsigned __int128)(n_ann + 1) * S128 >= (((unsigned __int128)1) << 63)) { set_error("skm_learn_sparse: n_ann * S does not fit 63 bits"); return SKM_ERR_UNSUPPORTED; }
    if (!d_nnz) { set_error("skm_learn_sparse: d_nnz is NULL"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_nnz, 0, 8, st));
    if (nseq == 0 || nres == 0 || n_ann == 0) return SKM_OK;
    if (nres >= (1ll << 31)) { set_error("skm_learn_sparse: more than 2^31 residues per call; split the shard"); return SKM_ERR_UNSUPPORTED; }
    if (!d_ann_id || !d_keys_out || !d_vals_out) { set_error("skm_learn_sparse: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_learn_sparse_workspace(nres);
    if (!workspace || workspace_bytes < need) { set_error("skm_learn_sparse: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(nres) * 8);
    uint64_t *keys_a = (uint64_t *)p, *keys_b = (uint64_t *)(p + seg);
    void *temp = p + 2 * seg;
    size_t temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    const uint64_t S = (uint64_t)S128;
    const uint64_t invalid = uint64_t(n_ann) * S;
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    int64_t grid = int64_t(sm_count()) * 8;
    const int64_t max_grid = (nres + SP_SEG - 1) / SP_SEG;
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    // positions outside [off[0], off[nseq]) are not written by the kernel
    SKM_CUDA_TRY(cudaMemsetAsync(keys_a, 0xFF, size_t(nres) * 8, st));
    SKM_CUDA_TRY(cudaFuncSetAttribute(window_keys_kernel<1, uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, sp_smem_bytes<uint64_t>()));
    window_keys_kernel<1, uint64_t><<<(unsigned)grid, TS_THREADS, sp_smem_bytes<uint64_t>(), st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k,
                                                                                      pow_k1, nullptr, d_ann_id, S, invalid, keys_a);
    SKM_LAUNCH_CHECK("window_keys_kernel<1>");
    // keys are < 2^end_bit except the all-ones fill, whose low bits are all ones too: it still sorts last
    const int end_bit = bits_for((unsigned __int128)invalid + 1);
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys_a, keys_b, nres, 0, end_bit, st));
    int64_t *num_runs = reinterpret_cast<int64_t *>(keys_a);     // keys_a is free after the sort
    temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceRunLengthEncode::Encode(temp, temp_bytes, keys_b, d_keys_out, d_vals_out, num_runs, (int)nres, st));
    coo_finish_kernel<<<1, 1, 0, st>>>(d_keys_out, num_runs, invalid, d_nnz);
    SKM_LAUNCH_CHECK("coo_finish_kernel");
    return SKM_OK;
}

// ---- wide learn: the matrix keyed by basis column (code spaces beyond the tables, up to 2^64 - 1) --------------
// Every window whose code the basis holds becomes the key a * K + col (skm_learn_sparse's key with the stride K of the
// basis in place of S); unannotated sequences get the rest row a = n_ann, so the column sums of the whole list are the
// Totals over all sequences (learn.smk:380) and the annotated matrix is the prefix key < n_ann * K.
size_t skm_learn_wide_workspace(int64_t nres) {
    using namespace skm;
    if (nres <= 0) return 256;
    return skm_learn_sparse_workspace(nres) + align256(SORTED_BUCKET_BYTES);
}

int skm_learn_wide(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                   const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t n_ann,
                   const uint64_t *d_sorted_codes, const int32_t *d_col_of_sorted, int64_t K,
                   uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_nnz, void *workspace,
                   size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    unsigned __int128 S128;
    int rc = wide_check(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, "skm_learn_wide", &S128);
    if (rc) return rc;
    if (n_ann < 0 || K < 0 || K >= (1ll << 31)) { set_error("skm_learn_wide: n_ann=%lld K=%lld outside [0, 2^31)", (long long)n_ann, (long long)K); return SKM_ERR_INVALID; }
    if ((unsigned __int128)(n_ann + 2) * (unsigned __int128)K >= ((unsigned __int128)1 << 63)) { set_error("skm_learn_wide: (n_ann + 2) * K does not fit 63 bits"); return SKM_ERR_UNSUPPORTED; }
    if (!d_nnz) { set_error("skm_learn_wide: d_nnz is NULL"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_nnz, 0, 8, st));
    if (nseq == 0 || nres == 0 || K == 0) return SKM_OK;
    if (!d_ann_id || !d_sorted_codes || !d_col_of_sorted || !d_keys_out || !d_vals_out) { set_error("skm_learn_wide: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_learn_wide_workspace(nres);
    if (!workspace || workspace_bytes < need) { set_error("skm_learn_wide: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(nres) * 8);
    uint64_t *keys_a = (uint64_t *)p, *keys_b = (uint64_t *)(p + seg);
    uint32_t *bucket = (uint32_t *)(p + 2 * seg);
    void *temp = p + 2 * seg + align256(SORTED_BUCKET_BYTES);
    size_t temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SortedBasis sb;
    rc = sorted_basis_init(&sb, d_sorted_codes, d_col_of_sorted, K, S128, bucket, st);
    if (rc) return rc;
    const uint64_t invalid = uint64_t(n_ann + 1) * uint64_t(K);
    uint64_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint64_t)nsym;
    int64_t grid = int64_t(sm_count()) * 8;
    const int64_t max_grid = (nres + SP_SEG - 1) / SP_SEG;
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    // positions outside [off[0], off[nseq]) are not written by the kernel
    SKM_CUDA_TRY(cudaMemsetAsync(keys_a, 0xFF, size_t(nres) * 8, st));
    SKM_CUDA_TRY(cudaFuncSetAttribute(learn_wide_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sp_smem_bytes<uint64_t>()));
    learn_wide_keys_kernel<<<(unsigned)grid, TS_THREADS, sp_smem_bytes<uint64_t>(), st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint64_t)nsym, k,
                                                                                      pow_k1, d_ann_id, n_ann, sb, invalid, keys_a);
    SKM_LAUNCH_CHECK("learn_wide_keys_kernel");
    // keys are < 2^end_bit except the all-ones fill, whose low bits are all ones too: it still sorts last
    const int end_bit = bits_for((unsigned __int128)invalid + 1);
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys_a, keys_b, nres, 0, end_bit, st));
    int64_t *num_runs = reinterpret_cast<int64_t *>(keys_a);     // keys_a is free after the sort
    temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceRunLengthEncode::Encode(temp, temp_bytes, keys_b, d_keys_out, d_vals_out, num_runs, (int)nres, st));
    coo_finish_kernel<<<1, 1, 0, st>>>(d_keys_out, num_runs, invalid, d_nnz);
    SKM_LAUNCH_CHECK("coo_finish_kernel");
    return SKM_OK;
}

// ---- grouped variant: 32-bit keys over a slice of annotations --------------------------------------------
// The caller has gathered the sequences of annotations [ann_lo, ann_lo + ann_n) into one contiguous batch
// (skm_gather_sequences), with ann_n * S < 2^32: keys fit 32 bits, the radix sort moves half the bytes per pass and
// needs only the bits of ann_n * S, and unannotated sequences never enter a sort.  The (key, count) runs are
// appended to the output at *d_nnz_inout as 64-bit global keys (ann_lo * S + key); groups processed in annotation
// order therefore leave one globally sorted COO list.
size_t skm_learn_sparse_group_workspace(int64_t nres) {
    using namespace skm;
    if (nres <= 0) return 256;
    size_t t_sort = 0, t_rle = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, t_sort, (const uint32_t *)nullptr, (uint32_t *)nullptr, nres, 0, 32);
    cub::DeviceRunLengthEncode::Encode(nullptr, t_rle, (const uint32_t *)nullptr, (uint32_t *)nullptr, (int32_t *)nullptr,
                                       (int64_t *)nullptr, (int)std::min<int64_t>(nres, (1ll << 31) - 1));
    return 4 * align256(size_t(nres) * 4) + align256(std::max(t_sort, t_rle)) + 1024;
}

namespace skm {
// out[base + i (+ shift)] = (key_base + uniq[i], counts[i]) for the runs below the invalid key; base = *nnz (entries this
// list holds so far).  With a placement (n_ins > 0) the list is written straight into a LARGER sorted list that also holds
// blocks other paths produce (the dense rows of the heavy annotations, skm_rows_emit): the block of annotation ins_ann[h]
// (ascending) has ins_cum[h] - ins_cum[h-1] entries, so an entry of annotation a moves up by ins_cum[#(ins_ann < a) - 1];
// ins_pos[h] (pre-set to INT64_MAX) receives the smallest index of THIS list that lies behind block h's predecessors —
// the caller's suffix-minimum over h turns it into where block h starts.  totals (nullable): += count per code.
struct Placement {
    const int64_t *ins_ann;     // [n_ins] ascending annotation ids of the blocks
    const int64_t *ins_cum;     // [n_ins] inclusive prefix of the block sizes
    long long *ins_pos;         // [n_ins]
    unsigned long long *totals; // [S] or NULL
    int n_ins;
};
__global__ void __launch_bounds__(256) coo_append_kernel(const uint32_t *__restrict__ uniq, const int32_t *__restrict__ counts,
                                                         const int64_t *__restrict__ num_runs, uint32_t invalid, uint64_t key_base,
                                                         const int64_t *__restrict__ nnz, int64_t capacity,
                                                         uint64_t *__restrict__ keys_out, int64_t *__restrict__ vals_out,
                                                         int64_t *__restrict__ n_new, uint32_t S, int64_t ann_lo, const Placement pl) {
    int64_t n = *num_runs;
    while (n > 0 && uniq[n - 1] >= invalid) --n;            // at most two trailing runs (invalid key, all-ones fill)
    const int64_t base = *nnz;
    if (pl.n_ins == 0 && base + n > capacity) n = capacity > base ? capacity - base : 0;      // the host checks the total afterwards
    auto blocks_before = [&](int64_t ann) {                 // #(ins_ann < ann)
        int lo = 0, hi = pl.n_ins;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(pl.ins_ann + mid) < ann) lo = mid + 1; else hi = mid; }
        return lo;
    };
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        const uint32_t u = uniq[i];
        int64_t o = base + i;
        if (pl.n_ins > 0 || pl.totals) {
            const uint32_t a_rel = u / S;
            if (pl.totals) atomicAdd(pl.totals + (u - a_rel * S), (unsigned long long)counts[i]);
            if (pl.n_ins > 0) {
                const int hb = blocks_before(ann_lo + a_rel);
                if (hb > 0) {
                    // first entry of this slice, or first entry behind a block boundary: a candidate for ins_pos[hb - 1]
                    if (i == 0 || blocks_before(ann_lo + uniq[i - 1] / S) != hb) atomicMin(pl.ins_pos + (hb - 1), (long long)(base + i));
                    o += __ldg(pl.ins_cum + hb - 1);
                }
            }
        }
        if (o < capacity) { keys_out[o] = key_base + u; vals_out[o] = counts[i]; }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_new = n;
}
__global__ void add_i64_kernel(int64_t *dst, const int64_t *src) { *dst += *src; }
}  // namespace skm

int skm_learn_sparse_group(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                           const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t ann_lo, int64_t ann_n,
                           uint64_t *d_keys_out, int64_t *d_vals_out, int64_t out_capacity, int64_t *d_nnz_inout,
                           void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    return skm_learn_sparse_group_place(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, d_ann_id, ann_lo, ann_n, d_keys_out, d_vals_out,
                                        out_capacity, d_nnz_inout, nullptr, nullptr, 0, nullptr, nullptr, workspace, workspace_bytes, stream);
}

int skm_learn_sparse_group_place(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                                 const uint8_t *d_lut, int nsym, int k, const int32_t *d_ann_id, int64_t ann_lo, int64_t ann_n,
                                 uint64_t *d_keys_out, int64_t *d_vals_out, int64_t out_capacity, int64_t *d_nnz_inout,
                                 const int64_t *d_ins_ann, const int64_t *d_ins_cum, int64_t n_ins, int64_t *d_ins_pos, int64_t *d_totals,
                                 void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (n_ins < 0 || n_ins > (1 << 30) || (n_ins > 0 && (!d_ins_ann || !d_ins_cum || !d_ins_pos))) { set_error("skm_learn_sparse_group_place: bad placement"); return SKM_ERR_INVALID; }
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    if (!ts_supported(nsym, k)) { set_error("skm_learn_sparse_group: nsym=%d k=%d outside the kernel envelope", nsym, k); return SKM_ERR_UNSUPPORTED; }
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (ann_lo < 0 || ann_n < 1 || ann_lo + ann_n > 0x7FFFFFFF || (unsigned __int128)ann_n * S128 >= (((unsigned __int128)1) << 32) - 1) {
        set_error("skm_learn_sparse_group: ann_n * nsym^k must stay below 2^32 - 1");
        return SKM_ERR_UNSUPPORTED;
    }
    if (!d_nnz_inout || out_capacity < 0) { set_error("skm_learn_sparse_group: bad output arguments"); return SKM_ERR_INVALID; }
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (nres >= (1ll << 31)) { set_error("skm_learn_sparse_group: more than 2^31 residues per call; split the group"); return SKM_ERR_UNSUPPORTED; }
    if (!d_ann_id || !d_keys_out || !d_vals_out) { set_error("skm_learn_sparse_group: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_learn_sparse_group_workspace(nres);
    if (!workspace || workspace_bytes < need) { set_error("skm_learn_sparse_group: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(nres) * 4);
    uint32_t *keys_a = (uint32_t *)p, *keys_b = (uint32_t *)(p + seg), *uniq = (uint32_t *)(p + 2 * seg);
    int32_t *counts = (int32_t *)(p + 3 * seg);
    void *temp = p + 4 * seg;
    const size_t temp_cap = workspace_bytes - size_t((char *)temp - (char *)workspace);
    size_t temp_bytes = temp_cap;
    const uint64_t S = (uint64_t)S128;
    const uint32_t invalid = uint32_t(uint64_t(ann_n) * S);
    uint32_t pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= (uint32_t)nsym;
    int64_t grid = int64_t(sm_count()) * 8;
    const int64_t max_grid = (nres + SP_SEG - 1) / SP_SEG;
    if (grid > max_grid) grid = max_grid < 1 ? 1 : max_grid;
    SKM_CUDA_TRY(cudaMemsetAsync(keys_a, 0xFF, size_t(nres) * 4, st));       // positions outside every sequence
    window_keys_kernel<1, uint32_t><<<(unsigned)grid, TS_THREADS, sp_smem_bytes<uint32_t>(), st>>>(d_residues, nres, d_offsets, nseq, d_lut, (uint32_t)nsym, k,
                                                                                      pow_k1, nullptr, d_ann_id, S, invalid, keys_a,
                                                                                      (int32_t)ann_lo, (int32_t)(ann_lo + ann_n));
    SKM_LAUNCH_CHECK("window_keys_kernel<1, u32>");
    const int end_bit = std::min(32, bits_for((unsigned __int128)invalid + 1));
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys_a, keys_b, nres, 0, end_bit, st));
    int64_t *num_runs = reinterpret_cast<int64_t *>(keys_a);                 // keys_a is free after the sort
    int64_t *n_new = num_runs + 1;
    temp_bytes = temp_cap;
    SKM_CUDA_TRY(cub::DeviceRunLengthEncode::Encode(temp, temp_bytes, keys_b, uniq, counts, num_runs, (int)nres, st));
    const int g2 = (int)std::min<int64_t>((nres + 255) / 256, int64_t(sm_count()) * 8);
    const Placement pl{d_ins_ann, d_ins_cum, reinterpret_cast<long long *>(d_ins_pos), reinterpret_cast<unsigned long long *>(d_totals), (int)n_ins};
    coo_append_kernel<<<g2, 256, 0, st>>>(uniq, counts, num_runs, invalid, uint64_t(ann_lo) * S, d_nnz_inout, out_capacity, d_keys_out, d_vals_out, n_new,
                                          (uint32_t)S, ann_lo, pl);
    SKM_LAUNCH_CHECK("coo_append_kernel");
    add_i64_kernel<<<1, 1, 0, st>>>(d_nnz_inout, n_new);
    SKM_LAUNCH_CHECK("add_i64_kernel");
    return SKM_OK;
}

size_t skm_coo_merge_workspace(int64_t n) {
    using namespace skm;
    if (n <= 0) return 256;
    size_t t_sort = 0, t_red = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t_sort, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const int64_t *)nullptr,
                                    (int64_t *)nullptr, n, 0, 64);
    cub::DeviceReduce::ReduceByKey(nullptr, t_red, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const int64_t *)nullptr,
                                   (int64_t *)nullptr, (int64_t *)nullptr, cub::Sum(), n);
    return 2 * align256(size_t(n) * 8) + align256(std::max(t_sort, t_red)) + 1024;
}

int skm_coo_merge(const uint64_t *d_keys_in, const int64_t *d_vals_in, int64_t n, uint64_t key_bound, uint64_t *d_keys_out,
                  int64_t *d_vals_out, int64_t *d_n_out, void *workspace, size_t workspace_bytes,
                  skm_stream_t stream) {
    using namespace skm;
    if (n < 0 || !d_n_out) { set_error("skm_coo_merge: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_n_out, 0, 8, st));
    if (n == 0) return SKM_OK;
    if (!d_keys_in || !d_vals_in || !d_keys_out || !d_vals_out) { set_error("skm_coo_merge: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_coo_merge_workspace(n);
    if (!workspace || workspace_bytes < need) { set_error("skm_coo_merge: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(n) * 8);
    uint64_t *sk = (uint64_t *)p;
    int64_t *sv = (int64_t *)(p + seg);
    void *temp = p + 2 * seg;
    size_t temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    // keys are < key_bound (0 = unknown): the sort only needs its bits (35 of 64 for the C3 matrix)
    const int end_bit = key_bound ? bits_for((unsigned __int128)key_bound) : 64;
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, d_keys_in, sk, d_vals_in, sv, n, 0, end_bit, st));
    temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceReduce::ReduceByKey(temp, temp_bytes, sk, d_keys_out, sv, d_vals_out, d_n_out, cub::Sum(), n, st));
    return SKM_OK;
}

// ---- Totals from the matrix -----------------------------------------------------------------------------------
// totals[code] += sum over annotations of M[ann, code]: the column sums of a COO list.  The learn step needs the
// k-mer totals over ALL sequences (learn.smk:380); the annotated part is already aggregated per (annotation, k-mer) in
// the matrix — one atomic per ENTRY instead of one per window — and only the unannotated sequences are still
// counted window by window (skm_basis_accumulate with d_first = NULL).
namespace skm {
__global__ void __launch_bounds__(256) coo_colsum_kernel(const uint64_t *__restrict__ keys, const int64_t *__restrict__ vals, int64_t nnz,
                                                         uint64_t S, unsigned long long *__restrict__ totals) {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nnz; i += int64_t(gridDim.x) * blockDim.x)
        atomicAdd(totals + keys[i] % S, (unsigned long long)vals[i]);
}
}  // namespace skm

int skm_coo_colsum(const uint64_t *d_keys, const int64_t *d_vals, int64_t nnz, int64_t S, int64_t *d_totals, skm_stream_t stream) {
    using namespace skm;
    if (nnz < 0 || S <= 0) { set_error("skm_coo_colsum: bad sizes"); return SKM_ERR_INVALID; }
    if (nnz == 0) return SKM_OK;
    if (!d_keys || !d_vals || !d_totals) { set_error("skm_coo_colsum: NULL argument"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>((nnz + 255) / 256, int64_t(sm_count()) * 16);
    coo_colsum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_keys, d_vals, nnz, (uint64_t)S, reinterpret_cast<unsigned long long *>(d_totals));
    SKM_LAUNCH_CHECK("coo_colsum_kernel");
    return SKM_OK;
}

// ---- merge of SORTED runs (the fan-in after the all_to_all: W runs, one per sending rank) ----------------------
// Pairwise merge tree (cub::DeviceMerge, ceil(log2 W) rounds of one streaming pass each) + reduce-by-key, instead of
// a radix sort over the key bits (5 passes for the C3 matrix).
size_t skm_coo_merge_runs_workspace(int64_t n, int n_runs) {
    using namespace skm;
    if (n <= 0 || n_runs <= 0) return 256;
    size_t t_m = 0, t_red = 0;
    const int half = (int)std::min<int64_t>(n, (1ll << 31) - 1);
    cub::DeviceMerge::MergePairs(nullptr, t_m, (const uint64_t *)nullptr, (const int64_t *)nullptr, half, (const uint64_t *)nullptr,
                                 (const int64_t *)nullptr, half, (uint64_t *)nullptr, (int64_t *)nullptr);
    cub::DeviceReduce::ReduceByKey(nullptr, t_red, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const int64_t *)nullptr,
                                   (int64_t *)nullptr, (int64_t *)nullptr, cub::Sum(), n);
    return 4 * align256(size_t(n) * 8) + align256(std::max(t_m, t_red)) + 1024;
}

int skm_coo_merge_runs(const uint64_t *d_keys_in, const int64_t *d_vals_in, const int64_t *run_offsets_host, int n_runs,
                       uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_n_out, void *workspace, size_t workspace_bytes,
                       skm_stream_t stream) {
    using namespace skm;
    if (n_runs < 0 || !d_n_out || (n_runs > 0 && !run_offsets_host)) { set_error("skm_coo_merge_runs: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_n_out, 0, 8, st));
    if (n_runs == 0) return SKM_OK;
    const int64_t base0 = run_offsets_host[0], n = run_offsets_host[n_runs] - base0;
    for (int r = 0; r < n_runs; ++r)
        if (run_offsets_host[r + 1] < run_offsets_host[r]) { set_error("skm_coo_merge_runs: run offsets must not decrease"); return SKM_ERR_INVALID; }
    if (n == 0) return SKM_OK;
    if (n >= (1ll << 31)) { set_error("skm_coo_merge_runs: more than 2^31 entries"); return SKM_ERR_UNSUPPORTED; }
    if (!d_keys_in || !d_vals_in || !d_keys_out || !d_vals_out) { set_error("skm_coo_merge_runs: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_coo_merge_runs_workspace(n, n_runs);
    if (!workspace || workspace_bytes < need) { set_error("skm_coo_merge_runs: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(n) * 8);
    uint64_t *kb[2] = {(uint64_t *)p, (uint64_t *)(p + seg)};
    int64_t *vb[2] = {(int64_t *)(p + 2 * seg), (int64_t *)(p + 3 * seg)};
    void *temp = p + 4 * seg;
    const size_t temp_cap = workspace_bytes - size_t((char *)temp - (char *)workspace);
    // run boundaries relative to the first run
    std::vector<int64_t> cur(n_runs + 1);
    for (int r = 0; r <= n_runs; ++r) cur[r] = run_offsets_host[r] - base0;
    const uint64_t *src_k = d_keys_in + base0;
    const int64_t *src_v = d_vals_in + base0;
    int flip = 0;
    while (cur.size() > 2) {
        std::vector<int64_t> next;
        next.push_back(0);
        uint64_t *dk = kb[flip];
        int64_t *dv = vb[flip];
        const int runs = int(cur.size()) - 1;
        for (int r = 0; r < runs; r += 2) {
            const int64_t a0 = cur[r], a1 = cur[r + 1];
            if (r + 1 < runs) {
                const int64_t b1 = cur[r + 2];
                size_t tb = temp_cap;
                SKM_CUDA_TRY(cub::DeviceMerge::MergePairs(temp, tb, src_k + a0, src_v + a0, (int)(a1 - a0), src_k + a1, src_v + a1, (int)(b1 - a1),
                                                          dk + a0, dv + a0, ::cuda::std::less<>{}, st));
                next.push_back(b1);
            } else {                                    // odd run out: carried over unchanged
                SKM_CUDA_TRY(cudaMemcpyAsync(dk + a0, src_k + a0, size_t(a1 - a0) * 8, cudaMemcpyDeviceToDevice, st));
                SKM_CUDA_TRY(cudaMemcpyAsync(dv + a0, src_v + a0, size_t(a1 - a0) * 8, cudaMemcpyDeviceToDevice, st));
                next.push_back(a1);
            }
        }
        cur.swap(next);
        src_k = dk; src_v = dv;
        flip ^= 1;
    }
    size_t tb = temp_cap;
    SKM_CUDA_TRY(cub::DeviceReduce::ReduceByKey(temp, tb, src_k, d_keys_out, src_v, d_vals_out, d_n_out, cub::Sum(), n, st));
    return SKM_OK;
}

// ---- packed exchange format: one 64-bit word per entry ---------------------------------------------------------------
// word = key << count_bits | count.  Halves the bytes of the multi-GPU exchange (all_to_all + merge tree move 8 instead of
// 16 bytes per entry) whenever the key (annotation * S + code) and the count fit 64 bits together; words sort like keys.
namespace skm {
__global__ void __launch_bounds__(256) coo_pack_kernel(const uint64_t *__restrict__ keys, const int64_t *__restrict__ vals, int64_t n,
                                                       int count_bits, uint64_t *__restrict__ out, int *__restrict__ overflow) {
    const uint64_t vmax = 1ull << count_bits, kmax = 1ull << (64 - count_bits);
    bool bad = false;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        const uint64_t k = keys[i], v = uint64_t(vals[i]);
        bad |= (v >= vmax) | (k >= kmax);
        out[i] = (k << count_bits) | (v & (vmax - 1));
    }
    if (bad) atomicOr(overflow, 1);
}
struct PackedKey {
    int bits;
    __host__ __device__ uint64_t operator()(uint64_t w) const { return w >> bits; }
};
struct PackedVal {
    uint64_t mask;
    __host__ __device__ int64_t operator()(uint64_t w) const { return int64_t(w & mask); }
};
}  // namespace skm

namespace skm {
// Sum the runs of equal keys of a SORTED list of packed words and unpack — the last step of the fan-in.  Two streaming
// passes (count the run heads per tile, then emit) instead of cub::DeviceReduce::ReduceByKey over transform iterators:
// a run is at most n_runs entries long (every incoming run has unique keys), so the head thread simply reads forward.
// 120 M words -> 93 M entries: 1.5 ms with CUB, ~0.6 ms here.
constexpr int PR_THREADS = 256, PR_PER = 8, PR_TILE = PR_THREADS * PR_PER;
// element (j, t) of a tile = tile_base + j * PR_THREADS + t: every load is coalesced (a lane's own 8 consecutive words
// would be 64 bytes apart from its neighbour's: 32 sectors per load instruction)
__global__ void __launch_bounds__(PR_THREADS) packed_heads_kernel(const uint64_t *__restrict__ w, int64_t n, int count_bits,
                                                                  int64_t *__restrict__ tile_heads) {
    const int64_t base = int64_t(blockIdx.x) * PR_TILE;
    int heads = 0;
#pragma unroll
    for (int j = 0; j < PR_PER; ++j) {
        const int64_t e = base + j * PR_THREADS + threadIdx.x;
        if (e < n) heads += (e == 0 || (w[e] >> count_bits) != (w[e - 1] >> count_bits)) ? 1 : 0;
    }
    __shared__ int s_w[PR_THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) heads += __shfl_xor_sync(FULL, heads, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = heads;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < PR_THREADS / 32; ++i) t += s_w[i];
        tile_heads[blockIdx.x] = t;
    }
}
__global__ void __launch_bounds__(PR_THREADS) packed_emit_kernel(const uint64_t *__restrict__ w, int64_t n, int count_bits,
                                                                 const int64_t *__restrict__ tile_off, int64_t n_tiles,
                                                                 uint64_t *__restrict__ keys_out, int64_t *__restrict__ vals_out,
                                                                 int64_t *__restrict__ n_out) {
    constexpr int NWP = PR_THREADS / 32;
    const uint64_t vmask = (1ull << count_bits) - 1;
    const int64_t base = int64_t(blockIdx.x) * PR_TILE;
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    __shared__ int s_cnt[PR_PER * NWP];          // heads of (row j, warp): element order = (j, warp, lane)
    __shared__ int s_off[PR_PER * NWP + 1];
    uint64_t word[PR_PER];
    unsigned bal[PR_PER];
#pragma unroll
    for (int j = 0; j < PR_PER; ++j) {
        const int64_t e = base + j * PR_THREADS + threadIdx.x;
        bool head = false;
        word[j] = 0;
        if (e < n) {
            word[j] = w[e];
            head = (e == 0) || (word[j] >> count_bits) != (w[e - 1] >> count_bits);
        }
        bal[j] = __ballot_sync(FULL, head);
        if (lane == 0) s_cnt[j * NWP + wp] = __popc(bal[j]);
    }
    __syncthreads();
    if (threadIdx.x < 32) {                       // exclusive scan of the 64 counters by one warp (two per lane)
        const int a0 = s_cnt[2 * lane], a1 = s_cnt[2 * lane + 1];
        int incl = a0 + a1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int x = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += x; }
        s_off[2 * lane] = incl - a0 - a1;
        s_off[2 * lane + 1] = incl - a1;
        if (lane == 31) s_off[PR_PER * NWP] = incl;
    }
    static_assert(PR_PER * NWP == 64, "the scan above handles 64 counters");
    __syncthreads();
    const int64_t t0 = tile_off[blockIdx.x];
#pragma unroll
    for (int j = 0; j < PR_PER; ++j) {
        if ((bal[j] >> lane) & 1u) {
            const int64_t e = base + j * PR_THREADS + threadIdx.x;
            const uint64_t k = word[j] >> count_bits;
            unsigned long long sum = word[j] & vmask;
            for (int64_t q = e + 1; q < n; ++q) {               // the rest of the run: at most one entry per incoming run
                const uint64_t x = w[q];
                if ((x >> count_bits) != k) break;
                sum += x & vmask;
            }
            const int64_t o = t0 + s_off[j * NWP + wp] + __popc(bal[j] & lt);
            keys_out[o] = k;
            vals_out[o] = (int64_t)sum;
        }
    }
    if (blockIdx.x == n_tiles - 1 && threadIdx.x == 0) *n_out = t0 + s_off[PR_PER * NWP];
}
}  // namespace skm

int skm_coo_pack(const uint64_t *d_keys, const int64_t *d_vals, int64_t n, int count_bits, uint64_t *d_packed, int *d_overflow,
                 skm_stream_t stream) {
    using namespace skm;
    if (n < 0 || count_bits < 1 || count_bits > 62 || !d_overflow) { set_error("skm_coo_pack: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_overflow, 0, sizeof(int), st));
    if (n == 0) return SKM_OK;
    if (!d_keys || !d_vals || !d_packed) { set_error("skm_coo_pack: NULL argument"); return SKM_ERR_INVALID; }
    coo_pack_kernel<<<(int)std::min<int64_t>((n + 255) / 256, int64_t(sm_count()) * 16), 256, 0, st>>>(d_keys, d_vals, n, count_bits, d_packed, d_overflow);
    SKM_LAUNCH_CHECK("coo_pack_kernel");
    return SKM_OK;
}

size_t skm_coo_merge_runs_packed_workspace(int64_t n, int n_runs) {
    using namespace skm;
    if (n <= 0 || n_runs <= 0) return 256;
    size_t t_m = 0, t_red = 0;
    const int half = (int)std::min<int64_t>(n, (1ll << 31) - 1);
    cub::DeviceMerge::MergeKeys(nullptr, t_m, (const uint64_t *)nullptr, half, (const uint64_t *)nullptr, half, (uint64_t *)nullptr);
    cub::TransformInputIterator<uint64_t, PackedKey, const uint64_t *> ki((const uint64_t *)nullptr, PackedKey{1});
    cub::TransformInputIterator<int64_t, PackedVal, const uint64_t *> vi((const uint64_t *)nullptr, PackedVal{1});
    cub::DeviceReduce::ReduceByKey(nullptr, t_red, ki, (uint64_t *)nullptr, vi, (int64_t *)nullptr, (int64_t *)nullptr, cub::Sum(), n);
    const size_t n_tiles = size_t((n + PR_TILE - 1) / PR_TILE);
    size_t t_scan = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, t_scan, (const int64_t *)nullptr, (int64_t *)nullptr, (int64_t)n_tiles);
    return 2 * align256(size_t(n) * 8) + align256(std::max(std::max(t_m, t_red), t_scan)) + 2 * align256(n_tiles * 8) + 1024;
}

int skm_coo_merge_runs_packed(const uint64_t *d_packed_in, const int64_t *run_offsets_host, int n_runs, int count_bits,
                              uint64_t *d_keys_out, int64_t *d_vals_out, int64_t *d_n_out, void *workspace, size_t workspace_bytes,
                              skm_stream_t stream) {
    using namespace skm;
    if (n_runs < 0 || !d_n_out || (n_runs > 0 && !run_offsets_host) || count_bits < 1 || count_bits > 62) { set_error("skm_coo_merge_runs_packed: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_n_out, 0, 8, st));
    if (n_runs == 0) return SKM_OK;
    const int64_t base0 = run_offsets_host[0], n = run_offsets_host[n_runs] - base0;
    for (int r = 0; r < n_runs; ++r)
        if (run_offsets_host[r + 1] < run_offsets_host[r]) { set_error("skm_coo_merge_runs_packed: run offsets must not decrease"); return SKM_ERR_INVALID; }
    if (n == 0) return SKM_OK;
    if (n >= (1ll << 31)) { set_error("skm_coo_merge_runs_packed: more than 2^31 entries"); return SKM_ERR_UNSUPPORTED; }
    if (!d_packed_in || !d_keys_out || !d_vals_out) { set_error("skm_coo_merge_runs_packed: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_coo_merge_runs_packed_workspace(n, n_runs);
    if (!workspace || workspace_bytes < need) { set_error("skm_coo_merge_runs_packed: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(n) * 8);
    uint64_t *kb[2] = {(uint64_t *)p, (uint64_t *)(p + seg)};
    void *temp = p + 2 * seg;
    const size_t temp_cap = workspace_bytes - size_t((char *)temp - (char *)workspace);
    std::vector<int64_t> cur(n_runs + 1);
    for (int r = 0; r <= n_runs; ++r) cur[r] = run_offsets_host[r] - base0;
    const uint64_t *src = d_packed_in + base0;
    int flip = 0;
    while (cur.size() > 2) {                              // pairwise merge tree over the packed words (they sort like keys)
        std::vector<int64_t> next;
        next.push_back(0);
        uint64_t *dk = kb[flip];
        const int runs = int(cur.size()) - 1;
        for (int r = 0; r < runs; r += 2) {
            const int64_t a0 = cur[r], a1 = cur[r + 1];
            if (r + 1 < runs) {
                const int64_t b1 = cur[r + 2];
                size_t tb = temp_cap;
                SKM_CUDA_TRY(cub::DeviceMerge::MergeKeys(temp, tb, src + a0, (int)(a1 - a0), src + a1, (int)(b1 - a1), dk + a0, ::cuda::std::less<>{}, st));
                next.push_back(b1);
            } else {
                SKM_CUDA_TRY(cudaMemcpyAsync(dk + a0, src + a0, size_t(a1 - a0) * 8, cudaMemcpyDeviceToDevice, st));
                next.push_back(a1);
            }
        }
        cur.swap(next);
        src = dk;
        flip ^= 1;
    }
    // reduce the runs of equal keys + unpack: count heads per tile, scan, emit (packed_heads_kernel / packed_emit_kernel)
    const int64_t n_tiles = (n + PR_TILE - 1) / PR_TILE;
    const size_t tiles_seg = align256(size_t(n_tiles) * 8);
    char *tail = reinterpret_cast<char *>(workspace) + workspace_bytes - 2 * tiles_seg - 256;
    tail = reinterpret_cast<char *>(reinterpret_cast<uintptr_t>(tail) & ~uintptr_t(255));
    int64_t *tile_heads = reinterpret_cast<int64_t *>(tail), *tile_off = reinterpret_cast<int64_t *>(tail + tiles_seg);
    packed_heads_kernel<<<(unsigned)n_tiles, PR_THREADS, 0, st>>>(src, n, count_bits, tile_heads);
    SKM_LAUNCH_CHECK("packed_heads_kernel");
    size_t tb = size_t(tail - (char *)temp);
    SKM_CUDA_TRY(cub::DeviceScan::ExclusiveSum(temp, tb, tile_heads, tile_off, n_tiles, st));
    packed_emit_kernel<<<(unsigned)n_tiles, PR_THREADS, 0, st>>>(src, n, count_bits, tile_off, n_tiles, d_keys_out, d_vals_out, d_n_out);
    SKM_LAUNCH_CHECK("packed_emit_kernel");
    return SKM_OK;
}

constexpr int64_t SKM_CSC_MAX_COLS = (1ll << 31) - 1;

size_t skm_csc_build_workspace_cols(int64_t nnz, int64_t n_ann, int64_t S) {
    using namespace skm;
    if (nnz <= 0) return 256 + align256(size_t(std::max<int64_t>(n_ann, 1)) * 8);
    size_t t_sort = 0, t_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t_sort, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const int64_t *)nullptr,
                                    (int64_t *)nullptr, nnz, 0, 64);
    // the colptr scan: sized for 2^27 columns, or for S + 1 beyond that
    const int64_t scan_n = std::max<int64_t>((int64_t)1 << 27, std::min<int64_t>(S, SKM_CSC_MAX_COLS) + 1);
    cub::DeviceScan::InclusiveSum(nullptr, t_scan, (const int64_t *)nullptr, (int64_t *)nullptr, scan_n);
    return 4 * align256(size_t(nnz) * 8) + align256(size_t(n_ann) * 8) + align256(std::max(t_sort, t_scan)) + 1024;
}

size_t skm_csc_build_workspace(int64_t nnz, int64_t n_ann) { return skm_csc_build_workspace_cols(nnz, n_ann, SKM_DENSE_MAX_SPACE); }

int skm_csc_build(const uint64_t *d_keys, const int64_t *d_vals, int64_t nnz, int64_t S, int64_t n_ann,
                  int64_t *d_colptr, int32_t *d_rows, int32_t *d_mvals, double *d_mnorm2, float *d_inv_m32,
                  int64_t *d_max_m, void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (nnz < 0 || S <= 0 || S > SKM_CSC_MAX_COLS || n_ann < 0 || !d_colptr) { set_error("skm_csc_build: bad arguments"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_colptr, 0, size_t(S + 1) * 8, st));
    if (d_mnorm2 && n_ann > 0) SKM_CUDA_TRY(cudaMemsetAsync(d_mnorm2, 0, size_t(n_ann) * 8, st));
    if (d_inv_m32 && n_ann > 0) SKM_CUDA_TRY(cudaMemsetAsync(d_inv_m32, 0, size_t(n_ann) * 4, st));
    if (d_max_m) SKM_CUDA_TRY(cudaMemsetAsync(d_max_m, 0, 8, st));
    if (nnz == 0) return SKM_OK;
    if (!d_keys || !d_vals || !d_rows || !d_mvals || !d_max_m) { set_error("skm_csc_build: NULL argument"); return SKM_ERR_INVALID; }
    const size_t need = skm_csc_build_workspace_cols(nnz, n_ann, S);
    if (!workspace || workspace_bytes < need) { set_error("skm_csc_build: workspace %zu < %zu", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    char *p = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    const size_t seg = align256(size_t(nnz) * 8);
    uint64_t *k_in = (uint64_t *)p, *k_out = (uint64_t *)(p + seg);
    int64_t *perm_in = (int64_t *)(p + 2 * seg), *perm_out = (int64_t *)(p + 3 * seg);
    unsigned long long *norm2 = (unsigned long long *)(p + 4 * seg);
    void *temp = p + 4 * seg + align256(size_t(n_ann) * 8);
    size_t temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    const int grid = (int)std::min<int64_t>((nnz + 255) / 256, int64_t(sm_count()) * 16);
    SKM_CUDA_TRY(cudaMemsetAsync(norm2, 0, size_t(n_ann) * 8, st));
    coo_row_norm2_kernel<<<grid, 256, 0, st>>>(d_keys, d_vals, nnz, (uint64_t)S, norm2);
    SKM_LAUNCH_CHECK("coo_row_norm2_kernel");
    csc_keys_kernel<<<grid, 256, 0, st>>>(d_keys, nnz, (uint64_t)S, (uint64_t)n_ann, k_in, perm_in);
    SKM_LAUNCH_CHECK("csc_keys_kernel");
    const int end_bit = bits_for((unsigned __int128)S * (unsigned __int128)std::max<int64_t>(n_ann, 1));
    SKM_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, k_in, k_out, perm_in, perm_out, nnz, 0, end_bit, st));
    csc_emit_kernel<<<grid, 256, 0, st>>>(k_out, perm_out, d_vals, nnz, (uint64_t)n_ann, d_rows, d_mvals,
                                          reinterpret_cast<unsigned long long *>(d_colptr), reinterpret_cast<unsigned long long *>(d_max_m));
    SKM_LAUNCH_CHECK("csc_emit_kernel");
    temp_bytes = workspace_bytes - size_t((char *)temp - (char *)workspace);
    SKM_CUDA_TRY(cub::DeviceScan::InclusiveSum(temp, temp_bytes, d_colptr, d_colptr, S + 1, st));
    if ((d_mnorm2 || d_inv_m32) && n_ann > 0) {
        norm2_finish_kernel<<<(int)std::min<int64_t>((n_ann + 255) / 256, 1024), 256, 0, st>>>(norm2, n_ann, d_mnorm2, d_inv_m32);
        SKM_LAUNCH_CHECK("norm2_finish_kernel");
    }
    return SKM_OK;
}

int skm_csc_pack(const int32_t *d_rows, const int32_t *d_mvals, int64_t nnz, uint32_t *d_packed, skm_stream_t stream) {
    using namespace skm;
    if (nnz < 0) { set_error("skm_csc_pack: negative size"); return SKM_ERR_INVALID; }
    if (nnz == 0) return SKM_OK;
    if (!d_rows || !d_mvals || !d_packed) { set_error("skm_csc_pack: NULL argument"); return SKM_ERR_INVALID; }
    csc_pack_kernel<<<(int)std::min<int64_t>((nnz + 255) / 256, int64_t(sm_count()) * 16), 256, 0, (cudaStream_t)stream>>>(d_rows, d_mvals, nnz, d_packed);
    SKM_LAUNCH_CHECK("csc_pack_kernel");
    return SKM_OK;
}

}  // extern "C"

namespace skm {
// the argument checks and the launch of skm_apply_sparse / skm_apply_sparse_rows
template <bool ROWS>
static int apply_sparse_launch(const char *fn, const int64_t *d_rowptr, const uint32_t *d_cols, const int32_t *d_vals, int64_t nq,
                               const int64_t *d_colptr, const int32_t *d_rows, const int32_t *d_mvals, const uint32_t *d_packed,
                               const double *d_mnorm2, const float *d_inv_m32, int64_t n_ann, int acc_bits, int32_t *d_top1,
                               int32_t *d_top2, double *d_score1, double *d_score2, double *d_qnorm2, double *d_out_rows,
                               int64_t ld_rows, skm_stream_t stream) {
    if (acc_bits != 32 && acc_bits != 64) { set_error("%s: acc_bits must be 32 or 64", fn); return SKM_ERR_INVALID; }
    const int64_t cap = (200 * 1024) / (acc_bits / 8);
    if (nq < 0 || n_ann <= 0 || n_ann > cap) { set_error("%s: n_ann=%lld outside [1, %lld] for %d-bit accumulators (shard the annotations)", fn, (long long)n_ann, (long long)cap, acc_bits); return n_ann > cap ? SKM_ERR_UNSUPPORTED : SKM_ERR_INVALID; }
    if (ROWS && ld_rows < n_ann) { set_error("%s: ld_rows=%lld < n_ann=%lld", fn, (long long)ld_rows, (long long)n_ann); return SKM_ERR_INVALID; }
    if (nq == 0) return SKM_OK;
    if (!d_rowptr || !d_colptr || !d_mnorm2 || !d_inv_m32 || !d_top1 || !d_top2 || !d_score1 || !d_score2 || (ROWS && !d_out_rows)) { set_error("%s: NULL argument", fn); return SKM_ERR_INVALID; }
    if (d_packed && n_ann > 65536 - 4 - SPA_DUMMY) { set_error("%s: the packed CSC holds 16-bit annotation indices (n_ann <= 65500)", fn); return SKM_ERR_INVALID; }
    if ((reinterpret_cast<uintptr_t>(d_inv_m32) & 15u) != 0) { set_error("%s: d_inv_m32 must be 16-byte aligned (vector loads)", fn); return SKM_ERR_INVALID; }
    const size_t smem = std::max<size_t>(size_t(n_ann + 4 + SPA_DUMMY) * (acc_bits / 8), 116 * 1024);   // > half an SM: one CTA per SM by construction
    const int grid = (int)std::min<int64_t>(nq, int64_t(sm_count()));
    cudaStream_t st = (cudaStream_t)stream;
#define SKM_LAUNCH_SPA(ACC, PK)                                                                                              \
    {                                                                                                                        \
        auto kern = apply_sparse_kernel<ACC, PK, ROWS>;                                                                      \
        SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                    \
        kern<<<grid, SPA_THREADS, smem, st>>>(d_rowptr, d_cols, d_vals, nq, d_colptr, d_rows, d_mvals, d_packed, d_mnorm2,   \
                                              d_inv_m32, (int)n_ann, d_top1, d_top2, d_score1, d_score2, d_qnorm2,           \
                                              d_out_rows, ld_rows);                                                          \
    }
    if (acc_bits == 32) { if (d_packed) SKM_LAUNCH_SPA(uint32_t, true) else SKM_LAUNCH_SPA(uint32_t, false) }
    else { if (d_packed) SKM_LAUNCH_SPA(unsigned long long, true) else SKM_LAUNCH_SPA(unsigned long long, false) }
#undef SKM_LAUNCH_SPA
    SKM_LAUNCH_CHECK("apply_sparse_kernel");
    return SKM_OK;
}
}  // namespace skm

extern "C" {

int skm_apply_sparse(const int64_t *d_rowptr, const uint32_t *d_cols, const int32_t *d_vals, int64_t nq,
                     const int64_t *d_colptr, const int32_t *d_rows, const int32_t *d_mvals, const uint32_t *d_packed, const double *d_mnorm2,
                     const float *d_inv_m32, int64_t n_ann, int acc_bits, int32_t *d_top1, int32_t *d_top2,
                     double *d_score1, double *d_score2, double *d_qnorm2, skm_stream_t stream) {
    return skm::apply_sparse_launch<false>("skm_apply_sparse", d_rowptr, d_cols, d_vals, nq, d_colptr, d_rows, d_mvals, d_packed,
                                           d_mnorm2, d_inv_m32, n_ann, acc_bits, d_top1, d_top2, d_score1, d_score2, d_qnorm2,
                                           nullptr, 0, stream);
}

int skm_apply_sparse_rows(const int64_t *d_rowptr, const uint32_t *d_cols, const int32_t *d_vals, int64_t nq,
                          const int64_t *d_colptr, const int32_t *d_rows, const int32_t *d_mvals, const uint32_t *d_packed,
                          const double *d_mnorm2, const float *d_inv_m32, int64_t n_ann, int acc_bits, int32_t *d_top1,
                          int32_t *d_top2, double *d_score1, double *d_score2, double *d_qnorm2, double *d_out_rows,
                          int64_t ld_rows, skm_stream_t stream) {
    return skm::apply_sparse_launch<true>("skm_apply_sparse_rows", d_rowptr, d_cols, d_vals, nq, d_colptr, d_rows, d_mvals, d_packed,
                                          d_mnorm2, d_inv_m32, n_ann, acc_bits, d_top1, d_top2, d_score1, d_score2, d_qnorm2,
                                          d_out_rows, ld_rows, stream);
}

}  // extern "C"
