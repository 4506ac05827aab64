// skm_csrsort.cu — per-sequence k-mer counts as CSR without a device-wide sort (kernel (b), sparse form).
//
// The first version of skm_count_csr wrote one key per residue to HBM and ran cub::DeviceSegmentedSort over the
// sequences: proteins (mean 350 residues) fall into CUB's "large segment" kernel, one 256-thread CTA per protein,
// and the step ran at 4 G keys/s — 15 ms per 200 k proteins, 1 % of the HBM roofline.  Here a WARP owns a sequence
// from the residue bytes to its finished CSR row:
//   scan     residues -> LUT -> symbols in the warp's shared buffer -> rolling codes (ts_group_walk, the scanner of
//            count_dense_warp_bytes_kernel); the key of every window (code, or basis column) goes to the warp's key buffer in shared memory;
//   sort     bitonic network, all compare-exchanges ascending (flip formulation), so n need not be a power of two:
//            partners at or beyond n act as +infinity.  32-bit keys of sequences up to 512 windows are sorted in
//            REGISTERS (16 keys per lane, shuffles for the cross-lane steps: 75 instructions per key instead of ~250),
//            everything else in shared memory;
//   encode   run heads -> (key, run length) written to the sequence's own slots of a temporary CSR
//            (tmp[off[s] + j]: a sequence never has more distinct k-mers than residues), distinct count -> rowcount.
// A scan of rowcount gives rowptr and a copy kernel compacts the rows.  HBM traffic: residues once, 8-12 B per
// distinct entry written, read and written again.  Sequences longer than the warp buffer (1024 windows; ~2 % of
// UniRef-like proteins) are queued and handled by one CTA each (8192 keys in shared memory; beyond that the network
// runs on a global scratch row).
// 64-bit keys (code spaces up to 2^64 - 1) use the same kernel; with a basis given as a sorted code list every
// temporary entry is looked up in a second, fully occupied pass (bucketed binary search) and the compaction drops the
// entries outside the basis.
#include <cub/cub.cuh>

#include "skm_common.cuh"
#include "skm_tile.cuh"

namespace skm {

constexpr int CS_WARPS = 8;                    // warps (= sequences in flight) per CTA of the warp kernel
constexpr int CS_KCAP_W = 1024;                // keys per warp buffer
constexpr int CS_REG_KEYS = 512;               // sequences up to this many windows are sorted in registers (16 keys per lane)
constexpr int CS_KCAP_C = 8192;                // keys per CTA buffer of the long-sequence kernel
constexpr int CS_LONG_THREADS = 256;

template <typename T> struct key_none;
template <> struct key_none<uint32_t> { static constexpr uint32_t v = 0xFFFFFFFFu; };
template <> struct key_none<uint64_t> { static constexpr uint64_t v = ~0ull; };

// ascending bitonic network over keys[0, n) by a group of GT threads (g = thread index in the group)
template <typename KeyT, int GT>
__device__ __forceinline__ void group_sort(KeyT *keys, int n, int g) {
    if (n < 2) return;
    int P = 2;
    while (P < n) P <<= 1;
    for (int k = 2; k <= P; k <<= 1) {
        const int hk = k >> 1;
        // flip step: i in the lower half of its k-block pairs with the mirrored element of the upper half
        for (int t = g; t < (P >> 1); t += GT) {
            const int blk = t / hk, r = t - blk * hk;
            const int i = blk * k + r, j = blk * k + (k - 1 - r);
            if (j < n) {
                const KeyT a = keys[i], b = keys[j];
                if (b < a) { keys[i] = b; keys[j] = a; }
            }
        }
        gsync<GT>();
        for (int d = hk >> 1; d > 0; d >>= 1) {
            for (int t = g; t < (P >> 1); t += GT) {
                const int i = ((t & ~(d - 1)) << 1) | (t & (d - 1)), j = i + d;
                if (j < n) {
                    const KeyT a = keys[i], b = keys[j];
                    if (b < a) { keys[i] = b; keys[j] = a; }
                }
            }
            gsync<GT>();
        }
    }
}

// ---- register-resident warp sort (sequences of up to 1024 windows) --------------------------------------------
// The network above costs ~11 SASS instructions per compare-exchange (two LDS, two STS, index arithmetic).  For the warp
// kernel the keys are instead held in registers, blocked: element i = lane * R + r lives in register r of `lane`
// (R = P / 32 for the padded size P).  Steps with distance < R are compare-exchanges between registers of one lane
// (one min + one max per pair); steps with distance >= R exchange with lane ^ (distance / R) by shuffle and keep the
// minimum or the maximum (2 instructions per key).  Same flip formulation, so everything is ascending and the
// all-ones padding / invalid key sorts last.  P = 512: 75 instructions per key against ~250 through shared memory.
__device__ __forceinline__ uint32_t shfl_xor_key(uint32_t v, int m) { return __shfl_xor_sync(FULL, v, m); }
__device__ __forceinline__ uint64_t shfl_xor_key(uint64_t v, int m) {
    const uint32_t lo = __shfl_xor_sync(FULL, uint32_t(v), m), hi = __shfl_xor_sync(FULL, uint32_t(v >> 32), m);
    return (uint64_t(hi) << 32) | lo;
}
__device__ __forceinline__ uint32_t shfl_up_key(uint32_t v) { return __shfl_up_sync(FULL, v, 1); }
__device__ __forceinline__ uint64_t shfl_up_key(uint64_t v) {
    const uint32_t lo = __shfl_up_sync(FULL, uint32_t(v), 1), hi = __shfl_up_sync(FULL, uint32_t(v >> 32), 1);
    return (uint64_t(hi) << 32) | lo;
}
template <typename KeyT> __device__ __forceinline__ void reg_ce(KeyT &a, KeyT &b) {
    const KeyT lo = a < b ? a : b, hi = a < b ? b : a;
    a = lo; b = hi;
}
// one half-cleaner step at distance 2^LD, then the smaller distances (compile-time recursion: every register index
// is a constant, so the key array stays in registers)
template <typename KeyT, int R, int LD>
__device__ __forceinline__ void sort_clean(KeyT (&key)[R], int lane) {
    if constexpr (LD >= 0) {
        constexpr int d = 1 << LD;
        if constexpr (d >= R) {                         // partner lane ^ (d / R), same register
            constexpr int m = d / R;
            const bool lower = (lane & m) == 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const KeyT o = shfl_xor_key(key[r], m), a = key[r];
                key[r] = lower ? (a < o ? a : o) : (a < o ? o : a);
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r)
                if ((r & d) == 0) reg_ce(key[r], key[r + d]);
        }
        sort_clean<KeyT, R, LD - 1>(key, lane);
    }
}
// stage k = 2^LK: flip step, half-cleaners, then the next stage up to 2^LOGP = 32 * R
template <typename KeyT, int R, int LK, int LOGP>
__device__ __forceinline__ void sort_stage(KeyT (&key)[R], int lane) {
    if constexpr (LK <= LOGP) {
        constexpr int k = 1 << LK;
        if constexpr (k <= R) {                         // flip inside a lane: t <-> k-1-t in every block of k registers
#pragma unroll
            for (int b0 = 0; b0 < R; b0 += k)
#pragma unroll
                for (int t = 0; t < k / 2; ++t) reg_ce(key[b0 + t], key[b0 + k - 1 - t]);
        } else {                                        // flip across lanes: (lane, r) <-> (mirrored lane, R-1-r)
            constexpr int L = k / R, m = L - 1;
            const bool lower = (lane & (L >> 1)) == 0;
            if constexpr (R == 1) {
                const KeyT o = shfl_xor_key(key[0], m), a = key[0];
                key[0] = lower ? (a < o ? a : o) : (a < o ? o : a);
            } else {
#pragma unroll
                for (int r = 0; r < R / 2; ++r) {
                    const KeyT o1 = shfl_xor_key(key[R - 1 - r], m), o2 = shfl_xor_key(key[r], m);
                    const KeyT a = key[r], c = key[R - 1 - r];
                    key[r] = lower ? (a < o1 ? a : o1) : (a < o1 ? o1 : a);
                    key[R - 1 - r] = lower ? (c < o2 ? c : o2) : (c < o2 ? o2 : c);
                }
            }
        }
        sort_clean<KeyT, R, LK - 2>(key, lane);
        sort_stage<KeyT, R, LK + 1, LOGP>(key, lane);
    }
}
template <typename KeyT, int R>
__device__ __forceinline__ void warp_sort_regs(KeyT (&key)[R], int lane) {
    constexpr int LOGP = (R == 1 ? 5 : R == 2 ? 6 : R == 4 ? 7 : R == 8 ? 8 : R == 16 ? 9 : 10);      // log2(32 * R)
    sort_stage<KeyT, R, 1, LOGP>(key, lane);
}

// padded index of key i in the warp's shared buffer: one spare word per 32 keeps both the scan's writes and the
// blocked reads (lane * R + r) spread over the banks
__device__ __forceinline__ int kpad(int i) { return i + (i >> 5); }

// keys[kpad(0 .. n)) (unsorted, invalid windows = NONE) -> sorted in registers -> run heads with their lengths written to
// tmp_keys / tmp_vals [b + slot]; returns the number of runs (= distinct valid keys).  Whole warp, converged.
template <typename KeyT, int R>
__device__ __forceinline__ int warp_sort_encode(const KeyT *keys, int n, int lane, int64_t b, KeyT *__restrict__ tmp_keys,
                                                int32_t *__restrict__ tmp_vals) {
    constexpr KeyT NONE = key_none<KeyT>::v;
    KeyT key[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = lane * R + r;
        key[r] = (i < n) ? keys[kpad(i)] : NONE;
    }
    warp_sort_regs<KeyT, R>(key, lane);
    // run heads; NONE keys are at the end
    const KeyT up = shfl_up_key(key[R - 1]);             // last key of the previous lane
    int nheads = 0, nvalid = 0, first_head = 0x7FFFFFFF;
    uint32_t headmask = 0;                              // bit r: register r starts a run (R <= 32)
    {
        const bool valid = key[0] != NONE;
        const bool head = valid && (lane == 0 || key[0] != up);
        nvalid += valid;
        if (head) { headmask |= 1u; first_head = lane * R; ++nheads; }
    }
#pragma unroll
    for (int r = 1; r < R; ++r) {
        const bool valid = key[r] != NONE;
        const bool head = valid && key[r] != key[r - 1];
        nvalid += valid;
        if (head) { headmask |= 1u << r; if (nheads == 0) first_head = lane * R + r; ++nheads; }
    }
    // exclusive prefix of the head counts (slot base of this lane) and the total
    int incl = nheads;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
    const int total = __shfl_sync(FULL, incl, 31);
    int tot_valid = nvalid;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot_valid += __shfl_xor_sync(FULL, tot_valid, o);
    // position of the next run head after this lane: suffix minimum of the lanes' first heads
    int suf = first_head;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_down_sync(FULL, suf, o); if (lane + o < 32 && t < suf) suf = t; }
    int next = __shfl_down_sync(FULL, suf, 1);
    if (lane == 31 || next == 0x7FFFFFFF) next = tot_valid;          // the last run ends where the valid keys end
    int slot = (incl - nheads) + nheads - 1;
#pragma unroll
    for (int r = R - 1; r >= 0; --r) {
        if (headmask & (1u << r)) {
            const int idx = lane * R + r;
            tmp_keys[b + slot] = key[r];
            tmp_vals[b + slot] = next - idx;
            next = idx;
            --slot;
        }
    }
    return total;
}

// MODE 0: key = code.  MODE 1: key = col_of_code[code] (table basis; filtered codes never enter).
// (A basis given as a sorted code list is applied afterwards by csr_lookup_kernel: a separate, fully occupied pass
// hides the latency of the dependent look-up loads that 24 sorting warps per SM could not.)
// LONG = false: one warp per sequence, sequences with more than kcap windows are appended to long_list.
// LONG = true : one CTA per queued sequence.
template <typename KeyT, int MODE, bool LONG>
__global__ void __launch_bounds__(LONG ? CS_LONG_THREADS : 32 * CS_WARPS)
csr_sort_kernel(const uint8_t *__restrict__ res, int64_t nres, const int64_t *__restrict__ off, int64_t nseq,
                const uint8_t *__restrict__ lut, KeyT nsym, int k, KeyT pow_k1, const int32_t *__restrict__ col_of_code,
                int kcap, int64_t *long_list, unsigned long long *n_long, KeyT *gscratch, int64_t gscratch_stride,
                KeyT *__restrict__ tmp_keys, int32_t *__restrict__ tmp_vals, int64_t *__restrict__ rowcount) {
    constexpr int GT = LONG ? CS_LONG_THREADS : 32;
    constexpr int SYM_BYTES = ts_sym_bytes(GT * TS_WALK_C);
    constexpr KeyT NONE = key_none<KeyT>::v;
    extern __shared__ __align__(128) uint8_t s_raw[];
    __shared__ uint8_t s_lut[256];
    __shared__ int s_wcnt[CS_LONG_THREADS / 32];
    const int grp = LONG ? 0 : (threadIdx.x >> 5);
    const int g = LONG ? int(threadIdx.x) : int(threadIdx.x & 31);
    const int lane = threadIdx.x & 31;
    const size_t key_bytes = size_t(LONG ? kcap : kcap + (kcap >> 5)) * sizeof(KeyT);      // warp buffers are padded (kpad)
    uint8_t *mine = s_raw + size_t(grp) * (key_bytes + SYM_BYTES);
    KeyT *s_key = reinterpret_cast<KeyT *>(mine);
    uint8_t *s_sym = mine + key_bytes;
    uint32_t sym_addr = smem_addr(s_sym);
    asm volatile("" : "+r"(sym_addr));
    ts_lut_init(s_lut, lut);
    __syncthreads();
    // ---- which sequences ----
    int64_t lo = 0, hi = 0;
    if (!LONG) {
        if (lane == 0) seq_range(off, nseq, int64_t(blockIdx.x) * CS_WARPS + grp, int64_t(gridDim.x) * CS_WARPS, &lo, &hi);
        lo = __shfl_sync(FULL, lo, 0);
        hi = __shfl_sync(FULL, hi, 0);
    } else {
        lo = blockIdx.x;
        hi = int64_t(*n_long);
    }
    for (int64_t it = lo; it < hi; it += (LONG ? int64_t(gridDim.x) : 1)) {
        const int64_t s = LONG ? long_list[it] : it;
        const int64_t b = __ldg(off + s), e = __ldg(off + s + 1);
        const int64_t L = e - b;
        const int n = (L >= k) ? int(L - (k - 1)) : 0;          // windows of the sequence
        if (n == 0) { if (g == 0) rowcount[s + 1] = 0; continue; }
        if (!LONG && n > kcap) {
            if (g == 0) long_list[atomicAdd(n_long, 1ull)] = s;
            continue;
        }
        KeyT *keys = (LONG && n > kcap) ? gscratch + int64_t(blockIdx.x) * gscratch_stride : s_key;
        // 32-bit keys of sequences up to 512 windows are sorted in registers (padded buffer layout); 64-bit keys stay on
        // the shared-memory network (twice the shuffles and 80 registers made the register version slower: 4.9 vs 3.8 ms)
        const bool in_regs = !LONG && sizeof(KeyT) == 4 && n <= CS_REG_KEYS;
        // ---- scan: key of window i (residues b + i .. b + i + k-1) goes to keys[i] ----
        ts_group_walk<GT, 2, KeyT>(res, nres, b, e, s_lut, s_sym, sym_addr, k, nsym, pow_k1, g, [&](int64_t widx, KeyT code, bool ok) {
            if (widx >= 0) {
                KeyT key = NONE;
                if (ok) {
                    if (MODE == 1) { const int32_t c = __ldg(col_of_code + code); if (c >= 0) key = KeyT(c); }
                    else key = code;
                }
                keys[in_regs ? int64_t(kpad(int(widx))) : widx] = key;
            }
        });
        int total = 0;
        if (sizeof(KeyT) == 4 && in_regs) {
            // ---- sort + encode in registers (one instantiation: several unrolled networks thrash the instruction cache) ----
            total = warp_sort_encode<KeyT, CS_REG_KEYS / 32>(keys, n, lane, b, tmp_keys, tmp_vals);
        } else {
        // ---- sort (shared / global memory network) ----
        group_sort<KeyT, GT>(keys, n, g);
        // ---- encode: run heads -> tmp[b + slot] ----
        for (int p0 = 0; p0 < n; p0 += GT) {
            const int p = p0 + g;
            KeyT key = NONE;
            bool head = false;
            int len = 0;
            if (p < n) {
                key = keys[p];
                head = key != NONE && (p == 0 || keys[p - 1] != key);
                if (head) {
                    int q = p + 1;
                    while (q < n && keys[q] == key) ++q;
                    len = q - p;
                }
            }
            const unsigned m = __ballot_sync(FULL, head);
            int slot = total + __popc(m & ((1u << lane) - 1u));
            int round = __popc(m);
            if (LONG) {
                if (lane == 0) s_wcnt[threadIdx.x >> 5] = round;
                __syncthreads();
                int before = 0, all = 0;
#pragma unroll
                for (int w = 0; w < CS_LONG_THREADS / 32; ++w) {
                    const int c = s_wcnt[w];
                    if (w < int(threadIdx.x >> 5)) before += c;
                    all += c;
                }
                slot += before;
                round = all;
                __syncthreads();
            }
            if (head) {
                tmp_keys[b + slot] = key;
                tmp_vals[b + slot] = len;
            }
            total += round;
        }
        }
        if (g == 0) rowcount[s + 1] = total;
        gsync<GT>();                        // the key buffer is rewritten by the next sequence
    }
}

// basis look-up of every temporary entry: tmp_cols[off[s] + j] = column of tmp_keys[off[s] + j] or -1;
// kept[s + 1] = entries of row s the basis holds.  One warp per row, one entry per lane: every lane runs its own
// (bucketed) binary search, 64 warps per SM hide the dependent loads.
__global__ void __launch_bounds__(256) csr_lookup_kernel(const int64_t *__restrict__ off, const int64_t *__restrict__ rowcount, int64_t nseq,
                                                         const uint64_t *__restrict__ tmp_keys, SortedBasis sb,
                                                         int32_t *__restrict__ tmp_cols, int64_t *__restrict__ kept) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    for (int64_t s = warp; s < nseq; s += nwarps) {
        const int64_t src = __ldg(off + s), cnt = rowcount[s + 1];
        int64_t n_kept = 0;
        for (int64_t j0 = 0; j0 < cnt; j0 += 32) {
            const int64_t j = j0 + lane;
            int32_t col = -1;
            if (j < cnt) { col = sorted_lookup(sb, tmp_keys[src + j]); tmp_cols[src + j] = col; }
            n_kept += __popc(__ballot_sync(FULL, col >= 0));
        }
        if (lane == 0) kept[s + 1] = n_kept;
    }
}

// out[rowptr[s] + j'] = tmp[off[s] + j] for the entries j < rowcount[s + 1] of row s (all of them, or with FILTER only
// those with tmp_cols >= 0, order preserved); one warp per row
template <typename KeyT, bool FILTER>
__global__ void __launch_bounds__(256) csr_compact_kernel(const int64_t *__restrict__ off, const int64_t *__restrict__ rowcount,
                                                          const int64_t *__restrict__ rowptr, int64_t nseq,
                                                          const KeyT *__restrict__ tmp_keys, const int32_t *__restrict__ tmp_cols,
                                                          const int32_t *__restrict__ tmp_vals, KeyT *__restrict__ keys_out,
                                                          uint32_t *__restrict__ cols_out, int32_t *__restrict__ vals_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    for (int64_t s = warp; s < nseq; s += nwarps) {
        const int64_t src = __ldg(off + s), cnt = rowcount[s + 1];
        int64_t dst = rowptr[s];
        for (int64_t j0 = 0; j0 < cnt; j0 += 32) {
            const int64_t j = j0 + lane;
            int32_t col = 0;
            bool keep = j < cnt;
            if (keep && FILTER) { col = tmp_cols[src + j]; keep = col >= 0; }
            const unsigned m = __ballot_sync(FULL, keep);
            if (keep) {
                const int64_t d = dst + __popc(m & ((1u << lane) - 1u));
                if (keys_out) keys_out[d] = tmp_keys[src + j];
                if (FILTER && cols_out) cols_out[d] = uint32_t(col);
                vals_out[d] = tmp_vals[src + j];
            }
            dst += __popc(m);
        }
    }
}

// bucket[q] = first index whose code >> shift is >= q  (q in [0, nbucket]); codes ascending
__global__ void __launch_bounds__(256) bucket_index_kernel(const uint64_t *__restrict__ codes, int64_t K, int shift, int64_t nbucket,
                                                           uint32_t *__restrict__ bucket) {
    for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q <= nbucket; q += int64_t(gridDim.x) * blockDim.x) {
        int64_t lo = 0, hi = K;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((codes[mid] >> shift) < uint64_t(q)) lo = mid + 1; else hi = mid;
        }
        bucket[q] = uint32_t(lo);
    }
}

int sorted_basis_init(SortedBasis *sb, const uint64_t *codes, const int32_t *col, int64_t K, unsigned __int128 S,
                      uint32_t *bucket, cudaStream_t st) {
    *sb = SortedBasis{codes, col, nullptr, K, 0};
    if (K <= 64) return SKM_OK;
    const int bits = bits_for(S);
    sb->shift = bits > SORTED_BUCKET_BITS ? bits - SORTED_BUCKET_BITS : 0;
    const int64_t nbucket = int64_t((S - 1) >> sb->shift) + 1;            // <= 2^20
    bucket_index_kernel<<<(int)std::min<int64_t>((nbucket + 256) / 256, 1024), 256, 0, st>>>(codes, K, sb->shift, nbucket, bucket);
    SKM_LAUNCH_CHECK("bucket_index_kernel");
    sb->bucket = bucket;
    return SKM_OK;
}

constexpr int64_t CS_MAX_RES = 1ll << 30;


struct CsPlan {
    size_t key_bytes;
    int long_grid;
    int64_t gscratch_stride;     // keys per CTA of the long kernel's global scratch (0: none needed)
    size_t tmp_keys, tmp_cols, tmp_vals, rowcount, kept, long_list, n_long, gscratch, bucket, scan_temp;
    size_t total;
};

static CsPlan cs_plan(int64_t nres, int64_t nseq, int64_t max_len, size_t key_bytes, bool with_cols, bool with_bucket) {
    CsPlan p{};
    p.key_bytes = key_bytes;
    p.long_grid = sm_count() * 2;
    p.gscratch_stride = (max_len > CS_KCAP_C) ? ((max_len + 31) & ~int64_t(31)) : 0;
    size_t t_scan = 0;
    cub::DeviceScan::InclusiveSum(nullptr, t_scan, (const int64_t *)nullptr, (int64_t *)nullptr, nseq + 1);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o += align256(bytes); return at; };
    p.tmp_keys = take(size_t(nres) * key_bytes);
    p.tmp_cols = take(with_cols ? size_t(nres) * 4 : 0);
    p.tmp_vals = take(size_t(nres) * 4);
    p.rowcount = take(size_t(nseq + 1) * 8);
    p.kept = take(with_cols ? size_t(nseq + 1) * 8 : 0);
    p.long_list = take(size_t(nseq) * 8);
    p.n_long = take(8);
    p.gscratch = take(size_t(p.gscratch_stride) * key_bytes * p.long_grid);
    p.bucket = take(with_bucket ? SORTED_BUCKET_BYTES : 0);
    p.scan_temp = take(t_scan);
    p.total = o + 512;
    return p;
}

template <typename KeyT, int MODE>
static int cs_run(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq, const uint8_t *d_lut, int nsym, int k,
                  const int32_t *d_col_of_code, const SortedBasis *sb, int64_t max_len, const CsPlan &pl, char *ws, int64_t *d_rowptr,
                  KeyT *d_keys_out, uint32_t *d_cols_out, int32_t *d_vals, cudaStream_t st) {
    KeyT pow_k1 = 1;
    for (int i = 0; i + 1 < k; ++i) pow_k1 *= KeyT(nsym);
    KeyT *tmp_keys = reinterpret_cast<KeyT *>(ws + pl.tmp_keys);
    int32_t *tmp_cols = sb ? reinterpret_cast<int32_t *>(ws + pl.tmp_cols) : nullptr;
    int32_t *tmp_vals = reinterpret_cast<int32_t *>(ws + pl.tmp_vals);
    int64_t *rowcount = reinterpret_cast<int64_t *>(ws + pl.rowcount);
    int64_t *long_list = reinterpret_cast<int64_t *>(ws + pl.long_list);
    unsigned long long *n_long = reinterpret_cast<unsigned long long *>(ws + pl.n_long);
    KeyT *gscratch = pl.gscratch_stride ? reinterpret_cast<KeyT *>(ws + pl.gscratch) : nullptr;
    SKM_CUDA_TRY(cudaMemsetAsync(n_long, 0, 8, st));
    SKM_CUDA_TRY(cudaMemsetAsync(rowcount, 0, 8, st));
    // warp kernel
    {
        constexpr int SYM_W = ts_sym_bytes(32 * TS_WALK_C);
        const size_t smem = size_t(CS_WARPS) * (size_t(CS_KCAP_W + (CS_KCAP_W >> 5)) * sizeof(KeyT) + SYM_W);
        auto kern = csr_sort_kernel<KeyT, MODE, false>;
        SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = int((227 * 1024) / (smem + 1536));
        if (per_sm > 8) per_sm = 8;
        if (per_sm < 1) per_sm = 1;
        const int grid = (int)std::min<int64_t>((nseq + CS_WARPS - 1) / CS_WARPS, int64_t(sm_count()) * per_sm);
        kern<<<grid, 32 * CS_WARPS, smem, st>>>(d_residues, nres, d_offsets, nseq, d_lut, KeyT(nsym), k, pow_k1, d_col_of_code, CS_KCAP_W,
                                                 long_list, n_long, nullptr, 0, tmp_keys, tmp_vals, rowcount);
        SKM_LAUNCH_CHECK("csr_sort_kernel(warp)");
    }
    // long sequences (the list may be empty: the CTAs then exit at once)
    if (max_len - (k - 1) > CS_KCAP_W) {
        constexpr int SYM_C = ts_sym_bytes(CS_LONG_THREADS * TS_WALK_C);
        const size_t smem = size_t(CS_KCAP_C) * sizeof(KeyT) + SYM_C;
        auto kern = csr_sort_kernel<KeyT, MODE, true>;
        SKM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<pl.long_grid, CS_LONG_THREADS, smem, st>>>(d_residues, nres, d_offsets, nseq, d_lut, KeyT(nsym), k, pow_k1, d_col_of_code, CS_KCAP_C,
                                                           long_list, n_long, gscratch, pl.gscratch_stride, tmp_keys, tmp_vals, rowcount);
        SKM_LAUNCH_CHECK("csr_sort_kernel(long)");
    }
    const int64_t *counts = rowcount;
    if (sb) {
        int64_t *kept = reinterpret_cast<int64_t *>(ws + pl.kept);
        SKM_CUDA_TRY(cudaMemsetAsync(kept, 0, 8, st));
        csr_lookup_kernel<<<sm_count() * 8, 256, 0, st>>>(d_offsets, rowcount, nseq, reinterpret_cast<const uint64_t *>(tmp_keys), *sb, tmp_cols, kept);
        SKM_LAUNCH_CHECK("csr_lookup_kernel");
        counts = kept;
    }
    size_t temp_bytes = pl.total - pl.scan_temp;
    SKM_CUDA_TRY(cub::DeviceScan::InclusiveSum(ws + pl.scan_temp, temp_bytes, counts, d_rowptr, nseq + 1, st));
    if (sb) csr_compact_kernel<KeyT, true><<<sm_count() * 8, 256, 0, st>>>(d_offsets, rowcount, d_rowptr, nseq, tmp_keys, tmp_cols, tmp_vals, d_keys_out, d_cols_out, d_vals);
    else csr_compact_kernel<KeyT, false><<<sm_count() * 8, 256, 0, st>>>(d_offsets, rowcount, d_rowptr, nseq, tmp_keys, nullptr, tmp_vals, d_keys_out, nullptr, d_vals);
    SKM_LAUNCH_CHECK("csr_compact_kernel");
    return SKM_OK;
}

}  // namespace skm

extern "C" {

size_t skm_count_csr_sorted_workspace(int64_t nres, int64_t nseq, int64_t max_len, int key_bits) {
    using namespace skm;
    if (nres <= 0 || nseq <= 0) return 256;
    return cs_plan(nres, nseq, max_len, key_bits == 64 ? 8 : 4, key_bits == 64, key_bits == 64).total + 256;
}

int skm_count_csr_sorted(const uint8_t *d_residues, int64_t nres, const int64_t *d_offsets, int64_t nseq,
                         const uint8_t *d_lut, int nsym, int k, int key_bits, const int32_t *d_col_of_code, int64_t S,
                         const uint64_t *d_sorted_codes, const int32_t *d_col_of_sorted, int64_t K, int64_t max_len,
                         int64_t *d_rowptr, void *d_keys_out, uint32_t *d_cols_out, int32_t *d_vals, void *workspace,
                         size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    int rc = check_common(d_residues, nres, d_offsets, nseq, d_lut, nsym, k);
    if (rc) return rc;
    if (key_bits != 32 && key_bits != 64) { set_error("skm_count_csr_sorted: key_bits must be 32 or 64"); return SKM_ERR_INVALID; }
    if (!ts_supported(nsym, k)) { set_error("skm_count_csr_sorted: nsym=%d k=%d outside the kernel envelope", nsym, k); return SKM_ERR_UNSUPPORTED; }
    unsigned __int128 S128;
    code_space(nsym, k, &S128);
    if (key_bits == 32 && S128 >= ((unsigned __int128)1 << 32)) { set_error("skm_count_csr_sorted: nsym^k needs 64-bit keys"); return SKM_ERR_INVALID; }
    if (S128 > (((unsigned __int128)1 << 64) - 1)) { set_error("skm_count_csr_sorted: nsym^k = 2^64 collides with the invalid sentinel"); return SKM_ERR_UNSUPPORTED; }
    if (d_col_of_code && (key_bits != 32 || (unsigned __int128)S != S128)) { set_error("skm_count_csr_sorted: a column table needs 32-bit keys and S = nsym^k"); return SKM_ERR_INVALID; }
    if (d_sorted_codes && (key_bits != 64 || !d_col_of_sorted || K < 0)) { set_error("skm_count_csr_sorted: a sorted basis needs 64-bit keys and its column map"); return SKM_ERR_INVALID; }
    if (d_cols_out && !d_sorted_codes) { set_error("skm_count_csr_sorted: d_cols_out needs a sorted basis"); return SKM_ERR_INVALID; }
    if (!d_rowptr) { set_error("skm_count_csr_sorted: d_rowptr is NULL"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    SKM_CUDA_TRY(cudaMemsetAsync(d_rowptr, 0, 8 * (size_t)(nseq + 1), st));
    if (nseq == 0 || nres == 0) return SKM_OK;
    if (!d_vals || (!d_keys_out && !d_cols_out)) { set_error("skm_count_csr_sorted: NULL output"); return SKM_ERR_INVALID; }
    if (nres >= CS_MAX_RES || nseq >= (1ll << 31)) { set_error("skm_count_csr_sorted: more than 2^30 residues per call; split the shard"); return SKM_ERR_UNSUPPORTED; }
    if (max_len <= 0 || max_len > nres) max_len = nres;          // unknown: assume the worst
    const bool wide = key_bits == 64;
    const CsPlan pl = cs_plan(nres, nseq, max_len, wide ? 8 : 4, wide, wide);
    if (!workspace || workspace_bytes < pl.total + 256) { set_error("skm_count_csr_sorted: workspace %zu < %zu", workspace_bytes, pl.total + 256); return SKM_ERR_WORKSPACE; }
    char *ws = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    SortedBasis sb{};
    if (wide && d_sorted_codes) {
        rc = sorted_basis_init(&sb, d_sorted_codes, d_col_of_sorted, K, S128, reinterpret_cast<uint32_t *>(ws + pl.bucket), st);
        if (rc) return rc;
    }
    if (!wide) {
        if (d_col_of_code) return cs_run<uint32_t, 1>(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, d_col_of_code, nullptr, max_len, pl, ws, d_rowptr, (uint32_t *)d_keys_out, nullptr, d_vals, st);
        return cs_run<uint32_t, 0>(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, nullptr, nullptr, max_len, pl, ws, d_rowptr, (uint32_t *)d_keys_out, nullptr, d_vals, st);
    }
    return cs_run<uint64_t, 0>(d_residues, nres, d_offsets, nseq, d_lut, nsym, k, nullptr, d_sorted_codes ? &sb : nullptr, max_len, pl, ws, d_rowptr, (uint64_t *)d_keys_out, d_cols_out, d_vals, st);
}

}  // extern "C"
