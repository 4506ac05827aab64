// skm_csv.cu — the reference's CSV interchange files formatted on the device: only text crosses PCIe.
//
//   float64 cells      shortest round-trip decimal, printed the way pyarrow's CSV writer prints a double (the
//                      seq-annotation-scores files of apply.smk:295-299 and learn.smk:821-849): Ryu's shortest digits
//                      (Adams, PLDI 2018; tables in skm_csv_pow5.cuh), decimal notation for exponents -6 .. 9,
//                      d[.ddd]e±x otherwise, "nan" / "inf" / "-inf" / "-0".
//   association rows   A cells and the row label quoted as pyarrow quotes strings ("..." with inner quotes doubled);
//                      the full cosine block of a query chunk, or the top-2-masked rows of eval_apply
//                      (learn.smk:831-849: the two best scores, "nan" elsewhere) straight from the top-2.
//   count rows         CSR over the file's k-mer columns in the two layouts of the reference: learn.smk:328-357 (label
//                      first, pre-escaped by the caller; zeros blank) and learn.smk:583-594 (zeros "0", label last
//                      and quoted).
//
// Every writer is two passes: *_measure gives each row's byte length and scans them into row offsets (relative to the
// first row), the writer then puts each row at its offset.  One warp per association row (cells in groups of 32, a
// warp scan places them); one CTA per count row walking the K columns in tiles, the nonzeros of a tile dropped into
// shared memory and a block scan placing every cell.
#include <cub/cub.cuh>

#include "skm_common.cuh"
#include "skm_csv_pow5.cuh"

namespace skm {

__device__ const uint64_t g_pow5_inv[SKM_POW5_INV_SIZE][2] = SKM_POW5_INV_SPLIT_INIT;
__device__ const uint64_t g_pow5[SKM_POW5_SIZE][2] = SKM_POW5_SPLIT_INIT;
#ifndef __CUDA_ARCH__
static const uint64_t h_pow5_inv[SKM_POW5_INV_SIZE][2] = SKM_POW5_INV_SPLIT_INIT;
static const uint64_t h_pow5[SKM_POW5_SIZE][2] = SKM_POW5_SPLIT_INIT;
#endif

__host__ __device__ __forceinline__ uint32_t pow5bits(int32_t e) { return uint32_t(((uint32_t)e * 1217359u) >> 19) + 1; }
__host__ __device__ __forceinline__ uint32_t log10pow2(int32_t e) { return ((uint32_t)e * 78913u) >> 18; }
__host__ __device__ __forceinline__ uint32_t log10pow5(int32_t e) { return ((uint32_t)e * 732923u) >> 20; }

__host__ __device__ __forceinline__ uint32_t pow5factor(uint64_t v) {
    uint32_t n = 0;
    while (v % 5 == 0) { v /= 5; ++n; }
    return n;
}

// (m * mul) >> j for a 128-bit mul and j >= 64
__host__ __device__ __forceinline__ uint64_t mul_shift(uint64_t m, const uint64_t *mul, int32_t j) {
    const unsigned __int128 b0 = (unsigned __int128)m * mul[0];
    const unsigned __int128 b2 = (unsigned __int128)m * mul[1];
    return (uint64_t)(((b0 >> 64) + b2) >> (j - 64));
}

__host__ __device__ __forceinline__ void load_mul(bool inv, int idx, uint64_t out[2]) {
#ifdef __CUDA_ARCH__
    const uint64_t *p = inv ? g_pow5_inv[idx] : g_pow5[idx];
    out[0] = __ldg(p);
    out[1] = __ldg(p + 1);
#else
    const uint64_t *p = inv ? h_pow5_inv[idx] : h_pow5[idx];
    out[0] = p[0];
    out[1] = p[1];
#endif
}

// shortest decimal m * 10^e of a finite nonzero double (Ryu d2d, round-half-even on exact ties)
__host__ __device__ inline void d2d(uint64_t ieee_m, uint32_t ieee_e, uint64_t *out_m, int32_t *out_e) {
    int32_t e2;
    uint64_t m2;
    if (ieee_e == 0) { e2 = 1 - 1023 - 52 - 2; m2 = ieee_m; }
    else { e2 = int32_t(ieee_e) - 1023 - 52 - 2; m2 = (1ull << 52) | ieee_m; }
    const bool accept = (m2 & 1) == 0;
    const uint64_t mv = 4 * m2;
    const uint32_t mm_shift = (ieee_m != 0 || ieee_e <= 1) ? 1 : 0;
    uint64_t vr, vp, vm;
    int32_t e10;
    bool vm_tz = false, vr_tz = false;
    uint64_t mul[2];
    if (e2 >= 0) {
        const uint32_t q = log10pow2(e2) - (e2 > 3);
        e10 = int32_t(q);
        const int32_t k = SKM_POW5_INV_BITCOUNT + int32_t(pow5bits(int32_t(q))) - 1;
        const int32_t i = -e2 + int32_t(q) + k;
        load_mul(true, int(q), mul);
        vr = mul_shift(4 * m2, mul, i);
        vp = mul_shift(4 * m2 + 2, mul, i);
        vm = mul_shift(4 * m2 - 1 - mm_shift, mul, i);
        if (q <= 21) {
            if (mv % 5 == 0) vr_tz = pow5factor(mv) >= q;
            else if (accept) vm_tz = pow5factor(mv - 1 - mm_shift) >= q;
            else vp -= pow5factor(mv + 2) >= q;
        }
    } else {
        const uint32_t q = log10pow5(-e2) - (-e2 > 1);
        e10 = int32_t(q) + e2;
        const int32_t i = -e2 - int32_t(q);
        const int32_t k = int32_t(pow5bits(i)) - SKM_POW5_BITCOUNT;
        const int32_t j = int32_t(q) - k;
        load_mul(false, i, mul);
        vr = mul_shift(4 * m2, mul, j);
        vp = mul_shift(4 * m2 + 2, mul, j);
        vm = mul_shift(4 * m2 - 1 - mm_shift, mul, j);
        if (q <= 1) {
            vr_tz = true;
            if (accept) vm_tz = mm_shift == 1;
            else --vp;
        } else if (q < 63) {
            vr_tz = (mv & ((1ull << q) - 1)) == 0;
        }
    }
    int32_t removed = 0;
    uint8_t last = 0;
    uint64_t output;
    if (vm_tz || vr_tz) {
        while (vp / 10 > vm / 10) {
            vm_tz &= vm % 10 == 0;
            vr_tz &= last == 0;
            last = uint8_t(vr % 10);
            vr /= 10; vp /= 10; vm /= 10;
            ++removed;
        }
        if (vm_tz)
            while (vm % 10 == 0) {
                vr_tz &= last == 0;
                last = uint8_t(vr % 10);
                vr /= 10; vp /= 10; vm /= 10;
                ++removed;
            }
        if (vr_tz && last == 5 && vr % 2 == 0) last = 4;
        output = vr + ((vr == vm && (!accept || !vm_tz)) || last >= 5);
    } else {
        bool up = false;
        if (vp / 100 > vm / 100) { up = vr % 100 >= 50; vr /= 100; vp /= 100; vm /= 100; removed += 2; }
        while (vp / 10 > vm / 10) { up = vr % 10 >= 5; vr /= 10; vp /= 10; vm /= 10; ++removed; }
        output = vr + (vr == vm || up);
    }
    *out_m = output;
    *out_e = e10 + removed;
}

__host__ __device__ __forceinline__ int u64_len(uint64_t v) {
    int n = 1;
    while (v >= 10) { v /= 10; ++n; }
    return n;
}

__host__ __device__ __forceinline__ void put_u64(uint8_t *out, uint64_t v, int len) {
    for (int i = len - 1; i >= 0; --i) { out[i] = uint8_t('0' + v % 10); v /= 10; }
}

__host__ __device__ __forceinline__ int i64_len(int64_t v) {
    return v < 0 ? 1 + u64_len(0ull - uint64_t(v)) : u64_len(uint64_t(v));
}

__host__ __device__ __forceinline__ int put_i64(uint8_t *out, int64_t v) {
    if (v < 0) {
        *out = '-';
        const uint64_t u = 0ull - uint64_t(v);
        const int n = u64_len(u);
        put_u64(out + 1, u, n);
        return n + 1;
    }
    const int n = u64_len(uint64_t(v));
    put_u64(out, uint64_t(v), n);
    return n;
}

// A double as pyarrow's CSV writer prints it.  out == nullptr: the length only.  Returns the length (<= 25).
__host__ __device__ inline int fmt_f64(double v, uint8_t *out) {
    uint64_t bits;
    memcpy(&bits, &v, 8);
    const bool neg = bits >> 63;
    const uint64_t ieee_m = bits & ((1ull << 52) - 1);
    const uint32_t ieee_e = uint32_t(bits >> 52) & 0x7FFu;
    if (ieee_e == 0x7FFu) {
        if (ieee_m) { if (out) { out[0] = 'n'; out[1] = 'a'; out[2] = 'n'; } return 3; }
        int p = 0;
        if (out && neg) out[p] = '-';
        p += neg;
        if (out) { out[p] = 'i'; out[p + 1] = 'n'; out[p + 2] = 'f'; }
        return p + 3;
    }
    int p = 0;
    if (neg) { if (out) out[0] = '-'; p = 1; }
    if (ieee_e == 0 && ieee_m == 0) { if (out) out[p] = '0'; return p + 1; }
    uint64_t m;
    int32_t e;
    d2d(ieee_m, ieee_e, &m, &e);
    const int ol = u64_len(m);
    const int32_t x = e + ol - 1;                         // value = d.ddd * 10^x
    if (x >= -6 && x <= 9) {
        const int32_t dp = x + 1;                         // digits before the decimal point
        if (dp <= 0) {
            if (out) {
                out[p] = '0'; out[p + 1] = '.';
                for (int i = 0; i < -dp; ++i) out[p + 2 + i] = '0';
                put_u64(out + p + 2 - dp, m, ol);
            }
            return p + 2 - dp + ol;
        }
        if (dp >= ol) {
            if (out) {
                put_u64(out + p, m, ol);
                for (int i = ol; i < dp; ++i) out[p + i] = '0';
            }
            return p + dp;
        }
        if (out) {
            uint64_t lo = m, div = 1;
            for (int i = 0; i < ol - dp; ++i) div *= 10;
            put_u64(out + p, lo / div, dp);
            out[p + dp] = '.';
            put_u64(out + p + dp + 1, lo % div, ol - dp);
        }
        return p + ol + 1;
    }
    const uint32_t ax = uint32_t(x < 0 ? -x : x);
    const int xl = u64_len(ax);
    const int n = p + ol + (ol > 1) + 2 + xl;
    if (out) {
        if (ol > 1) {
            uint64_t div = 1;
            for (int i = 0; i < ol - 1; ++i) div *= 10;
            out[p] = uint8_t('0' + m / div);
            out[p + 1] = '.';
            put_u64(out + p + 2, m % div, ol - 1);
        } else {
            out[p] = uint8_t('0' + m);
        }
        const int q = p + ol + (ol > 1);
        out[q] = 'e';
        out[q + 1] = x < 0 ? '-' : '+';
        put_u64(out + q + 2, ax, xl);
    }
    return n;
}

// pyarrow's quoting of a string cell: "..." with every inner '"' doubled
__device__ __forceinline__ int64_t quoted_len(const uint8_t *s, int64_t n, int lane) {
    int64_t q = 0;
    for (int64_t i = lane; i < n; i += 32) q += s[i] == '"';
    for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(FULL, q, o);
    return n + q + 2;
}

__device__ __forceinline__ int64_t put_quoted(uint8_t *out, const uint8_t *s, int64_t n) {
    int64_t p = 0;
    out[p++] = '"';
    for (int64_t i = 0; i < n; ++i) {
        const uint8_t c = s[i];
        out[p++] = c;
        if (c == '"') out[p++] = '"';
    }
    out[p++] = '"';
    return p;
}

// ---- association rows ------------------------------------------------------------------------------------------------
struct FullCells {
    const double *scores;
    int64_t ld;
    __device__ __forceinline__ double operator()(int64_t r, int64_t j) const { return __ldg(scores + r * ld + j); }
};

struct Top2Cells {
    const int32_t *top1, *top2;
    const double *s1, *s2;
    __device__ __forceinline__ double operator()(int64_t r, int64_t j) const {
        if (j == __ldg(top2 + r)) return __ldg(s2 + r);
        if (j == __ldg(top1 + r)) return __ldg(s1 + r);
        return __longlong_as_double(0x7FF8000000000000ll);
    }
};

constexpr int CSV_WARPS = 8;

template <class Cells>
__global__ void __launch_bounds__(CSV_WARPS * 32) assoc_measure_kernel(Cells cells, int64_t rows, int64_t A, const uint8_t *__restrict__ labels,
                                                                       const int64_t *__restrict__ lab_off, int64_t *__restrict__ row_bytes) {
    const int lane = threadIdx.x & 31;
    for (int64_t r = int64_t(blockIdx.x) * CSV_WARPS + (threadIdx.x >> 5); r < rows; r += int64_t(gridDim.x) * CSV_WARPS) {
        int64_t n = 0;
        for (int64_t j = lane; j < A; j += 32) n += fmt_f64(cells(r, j), nullptr) + 1;
        for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(FULL, n, o);
        const int64_t l0 = lab_off[r];
        n += quoted_len(labels + l0, lab_off[r + 1] - l0, lane) + 1;
        if (lane == 0) row_bytes[r] = n;
    }
}

template <class Cells>
__global__ void __launch_bounds__(CSV_WARPS * 32) assoc_write_kernel(Cells cells, int64_t rows, int64_t A, const uint8_t *__restrict__ labels,
                                                                     const int64_t *__restrict__ lab_off, const int64_t *__restrict__ row_off,
                                                                     uint8_t *__restrict__ text) {
    const int lane = threadIdx.x & 31;
    const int64_t base0 = row_off[0];
    for (int64_t r = int64_t(blockIdx.x) * CSV_WARPS + (threadIdx.x >> 5); r < rows; r += int64_t(gridDim.x) * CSV_WARPS) {
        uint8_t *out = text + (row_off[r] - base0);
        int64_t pos = 0;
        for (int64_t j0 = 0; j0 < A; j0 += 32) {
            const int64_t j = j0 + lane;
            const double v = j < A ? cells(r, j) : 0.0;
            const int len = j < A ? fmt_f64(v, nullptr) + 1 : 0;
            int incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += t; }
            if (j < A) {
                uint8_t *c = out + pos + (incl - len);
                fmt_f64(v, c);
                c[len - 1] = ',';
            }
            pos += __shfl_sync(FULL, incl, 31);
        }
        if (lane == 0) {
            const int64_t l0 = lab_off[r];
            pos += put_quoted(out + pos, labels + l0, lab_off[r + 1] - l0);
            out[pos] = '\n';
        }
    }
}

// ---- count rows ------------------------------------------------------------------------------------------------------
constexpr int CNT_THREADS = 256;

__global__ void __launch_bounds__(CSV_WARPS * 32) counts_measure_kernel(const int64_t *__restrict__ rowptr, const int64_t *__restrict__ vals,
                                                                        int64_t rows, int64_t K, const int64_t *__restrict__ seq_count,
                                                                        const int64_t *__restrict__ kmer_count, const uint8_t *__restrict__ labels,
                                                                        const int64_t *__restrict__ lab_off, int layout,
                                                                        int64_t *__restrict__ row_bytes) {
    const int lane = threadIdx.x & 31;
    for (int64_t r = int64_t(blockIdx.x) * CSV_WARPS + (threadIdx.x >> 5); r < rows; r += int64_t(gridDim.x) * CSV_WARPS) {
        const int64_t p0 = rowptr[r], p1 = rowptr[r + 1];
        int64_t n = 0, nz = 0;
        for (int64_t i = p0 + lane; i < p1; i += 32) {
            const int64_t v = vals[i];
            if (v) { n += i64_len(v); ++nz; }
        }
        for (int o = 16; o; o >>= 1) { n += __shfl_xor_sync(FULL, n, o); nz += __shfl_xor_sync(FULL, nz, o); }
        const int64_t sc = seq_count[r], kc = kmer_count[r], l0 = lab_off[r], ln = lab_off[r + 1] - l0;
        n += K + 1;                                                  // a ',' before every k-mer cell, the '\n'
        if (layout == 0) {
            n += ln + 2 + (sc ? i64_len(sc) : 0) + (kc ? i64_len(kc) : 0);
        } else {
            n += (K - nz) + i64_len(sc) + 1 + i64_len(kc) + 1 + quoted_len(labels + l0, ln, lane);
        }
        if (lane == 0) row_bytes[r] = n;
    }
}

// one CTA per row: the K cells in tiles of CNT_THREADS columns; a tile's nonzeros are the next ones of the row whose
// column falls in the tile (columns ascending), their lengths go to shared memory and a block scan places every cell
__global__ void __launch_bounds__(CNT_THREADS) counts_write_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ cols,
                                                                   const int64_t *__restrict__ vals, int64_t rows, int64_t K,
                                                                   const int64_t *__restrict__ seq_count, const int64_t *__restrict__ kmer_count,
                                                                   const uint8_t *__restrict__ labels, const int64_t *__restrict__ lab_off,
                                                                   int layout, const int64_t *__restrict__ row_off, uint8_t *__restrict__ text) {
    using Scan = cub::BlockScan<int, CNT_THREADS>;
    __shared__ typename Scan::TempStorage s_scan;
    __shared__ int64_t s_val[CNT_THREADS];
    const int t = threadIdx.x;
    const int64_t base0 = row_off[0];
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
        uint8_t *out = text + (row_off[r] - base0);
        const int64_t sc = seq_count[r], kc = kmer_count[r], l0 = lab_off[r], ln = lab_off[r + 1] - l0;
        int64_t pos = 0;
        if (layout == 0) {
            for (int64_t i = t; i < ln; i += CNT_THREADS) out[i] = labels[l0 + i];
            pos = ln;                                               // every thread follows pos, thread 0 writes
            if (t == 0) out[pos] = ',';
            ++pos;
            if (t == 0 && sc) put_i64(out + pos, sc);
            pos += sc ? i64_len(sc) : 0;
            if (t == 0) out[pos] = ',';
            ++pos;
            if (t == 0 && kc) put_i64(out + pos, kc);
            pos += kc ? i64_len(kc) : 0;
        } else {
            if (t == 0) put_i64(out, sc);
            pos = i64_len(sc);
            if (t == 0) out[pos] = ',';
            ++pos;
            if (t == 0) put_i64(out + pos, kc);
            pos += i64_len(kc);
        }
        int64_t p = rowptr[r];
        const int64_t p1 = rowptr[r + 1];
        for (int64_t c0 = 0; c0 < K; c0 += CNT_THREADS) {
            s_val[t] = 0;
            __syncthreads();
            const int64_t i = p + t;
            const bool in = i < p1 && int64_t(cols[i]) >= c0 && int64_t(cols[i]) < c0 + CNT_THREADS;
            if (in) s_val[cols[i] - c0] = vals[i];
            const int taken = __syncthreads_count(in);
            p += taken;
            const int64_t c = c0 + t;
            const int64_t v = s_val[t];
            const int len = c < K ? 1 + (v ? i64_len(v) : layout) : 0;
            int excl, total;
            Scan(s_scan).ExclusiveSum(len, excl, total);
            if (c < K) {
                uint8_t *o = out + pos + excl;
                o[0] = ',';
                if (v) put_i64(o + 1, v);
                else if (layout) o[1] = '0';
            }
            pos += total;
            __syncthreads();
        }
        if (layout == 1 && t == 0) {
            out[pos++] = ',';
            pos += put_quoted(out + pos, labels + l0, ln);
        }
        if (t == 0) out[pos] = '\n';                               // thread 0 alone holds pos past the label
        __syncthreads();
    }
}

inline int grid_for(int64_t items, int per_block) {
    int64_t g = (items + per_block - 1) / per_block;
    const int64_t cap = int64_t(sm_count()) * 32;
    if (g > cap) g = cap;
    return int(g < 1 ? 1 : g);
}

// row_off[0] = 0, row_off[1..rows] = inclusive sum of row_bytes (workspace: row_bytes then cub's scratch)
inline size_t scan_temp_bytes(int64_t rows) {
    size_t temp = 0;
    cub::DeviceScan::InclusiveSum(nullptr, temp, (const int64_t *)nullptr, (int64_t *)nullptr, rows);
    return temp;
}

inline size_t rows_workspace(int64_t rows) { return align256(size_t(rows > 0 ? rows : 1) * 8) + align256(scan_temp_bytes(rows > 0 ? rows : 1)); }

inline int scan_rows(int64_t *row_bytes, int64_t rows, int64_t *row_off, void *ws, size_t ws_bytes, cudaStream_t st) {
    SKM_CUDA_TRY(cudaMemsetAsync(row_off, 0, sizeof(int64_t), st));
    if (rows == 0) return SKM_OK;
    size_t temp = scan_temp_bytes(rows);
    void *scratch = static_cast<uint8_t *>(ws) + align256(size_t(rows) * 8);
    SKM_CUDA_TRY(cub::DeviceScan::InclusiveSum(scratch, temp, row_bytes, row_off + 1, rows, st));
    return SKM_OK;
}

inline int check_rows_ws(const char *who, int64_t rows, void *ws, size_t ws_bytes) {
    if (ws_bytes < rows_workspace(rows) || (!ws && rows > 0)) {
        set_error("%s: workspace of %zu bytes, %zu needed", who, ws_bytes, rows_workspace(rows));
        return SKM_ERR_WORKSPACE;
    }
    return SKM_OK;
}

template <class Cells>
int assoc_measure(const char *who, Cells cells, int64_t rows, int64_t A, const uint8_t *labels, const int64_t *lab_off, int64_t *row_off,
                  void *ws, size_t ws_bytes, cudaStream_t st) {
    if (rows < 0 || A < 0 || !row_off || (rows > 0 && !lab_off)) { set_error("%s: bad sizes or NULL argument", who); return SKM_ERR_INVALID; }
    int rc = check_rows_ws(who, rows, ws, ws_bytes);
    if (rc) return rc;
    if (rows > 0) {
        assoc_measure_kernel<<<grid_for(rows, CSV_WARPS), CSV_WARPS * 32, 0, st>>>(cells, rows, A, labels, lab_off, (int64_t *)ws);
        SKM_LAUNCH_CHECK(who);
    }
    return scan_rows((int64_t *)ws, rows, row_off, ws, ws_bytes, st);
}

template <class Cells>
int assoc_write(const char *who, Cells cells, int64_t rows, int64_t A, const uint8_t *labels, const int64_t *lab_off, const int64_t *row_off,
                uint8_t *text, cudaStream_t st) {
    if (rows < 0 || A < 0) { set_error("%s: bad sizes", who); return SKM_ERR_INVALID; }
    if (rows == 0) return SKM_OK;
    if (!lab_off || !row_off || !text) { set_error("%s: NULL argument", who); return SKM_ERR_INVALID; }
    assoc_write_kernel<<<grid_for(rows, CSV_WARPS), CSV_WARPS * 32, 0, st>>>(cells, rows, A, labels, lab_off, row_off, text);
    SKM_LAUNCH_CHECK(who);
    return SKM_OK;
}


// ---- count CSV parser ------------------------------------------------------------------------------------------------
// Quote parity: an inclusive XOR scan over the '"' bytes; a ',' or '\n' with parity 0 separates cells, a '\n' with
// parity 0 ends a row.  Then one CTA per row walks it in tiles of PARSE_THREADS x PARSE_BYTES bytes: every thread counts
// the separators in its bytes, a block scan gives each its field number and the position of the separator before it,
// and the thread owning a cell's closing separator parses the cell [previous separator + 1, separator).
constexpr int PARSE_THREADS = 256, PARSE_BYTES = 16;
constexpr unsigned long long PARSE_NO_ERROR = ~0ull;
constexpr uint32_t PARSE_FIELD_COUNT = 0xFFFFFFFFu;    // error field: the row has the wrong number of fields

struct IsQuote {
    __host__ __device__ __forceinline__ uint8_t operator()(uint8_t c) const { return c == '"'; }
};
struct XorOp {
    __host__ __device__ __forceinline__ uint8_t operator()(uint8_t a, uint8_t b) const { return a ^ b; }
};
struct RowEnd {
    const uint8_t *text, *parity;
    __host__ __device__ __forceinline__ bool operator()(int64_t i) const { return text[i] == '\n' && parity[i] == 0; }
};
struct MaxOp {
    __device__ __forceinline__ int64_t operator()(int64_t a, int64_t b) const { return a > b ? a : b; }
};

// the cell grammar: empty (0), [0-9]+, [0-9]+\.0*, and d[.ddd]e[+-]x when the value is an integer below 2^63
__device__ __forceinline__ bool mul10_add(uint64_t &d, uint32_t x) {      // d = 10 d + x, false past 2^63 - 1
    if (d > (0x7FFFFFFFFFFFFFFFull - x) / 10) return false;
    d = d * 10 + x;
    return true;
}

__device__ __forceinline__ bool parse_count(const uint8_t *s, int64_t n, int64_t *out) {
    if (n == 0) { *out = 0; return true; }
    uint64_t d = 0;
    int64_t i = 0;
    int digits = 0, frac = 0, zeros = 0;      // zeros: fraction zeros not yet multiplied in
    while (i < n && s[i] >= '0' && s[i] <= '9') { if (!mul10_add(d, s[i] - '0')) return false; ++digits; ++i; }
    if (digits == 0) return false;
    if (i < n && s[i] == '.') {
        ++i;
        for (; i < n && s[i] >= '0' && s[i] <= '9'; ++i) {
            if (s[i] == '0') { ++zeros; continue; }
            for (; zeros > 0; --zeros, ++frac) if (!mul10_add(d, 0)) return false;
            if (!mul10_add(d, s[i] - '0')) return false;
            ++frac;
        }
    }
    int ex = 0;
    if (i < n && s[i] == 'e') {
        ++i;
        bool neg = false;
        if (i < n && (s[i] == '+' || s[i] == '-')) { neg = s[i] == '-'; ++i; }
        int ed = 0;
        while (i < n && s[i] >= '0' && s[i] <= '9') { if (++ed > 3) return false; ex = ex * 10 + (s[i] - '0'); ++i; }
        if (ed == 0) return false;
        if (neg) ex = -ex;
    }
    if (i != n) return false;
    for (int shift = ex - frac; shift != 0;) {
        if (shift < 0) { if (d % 10) return false; d /= 10; ++shift; }
        else { if (!mul10_add(d, 0)) return false; --shift; }
    }
    *out = int64_t(d);
    return true;
}

template <bool WRITE>
__global__ void __launch_bounds__(PARSE_THREADS, 1) parse_cells_kernel(const uint8_t *__restrict__ text, const uint8_t *__restrict__ parity,
                                                                    const int64_t *__restrict__ row_start, const int64_t *__restrict__ row_end,
                                                                    int64_t rows, const int32_t *__restrict__ role, int nfields,
                                                                    const int64_t *__restrict__ entry_off, int64_t *__restrict__ row_nnz,
                                                                    int64_t *__restrict__ seq, int64_t *__restrict__ kc,
                                                                    int64_t *__restrict__ lab_start, int64_t *__restrict__ lab_end,
                                                                    int32_t *__restrict__ cols, int64_t *__restrict__ vals,
                                                                    unsigned long long *__restrict__ error) {
    using ScanI = cub::BlockScan<int, PARSE_THREADS>;
    using ScanL = cub::BlockScan<int64_t, PARSE_THREADS>;
    __shared__ typename ScanI::TempStorage s_si;
    __shared__ typename ScanL::TempStorage s_sl;
    const int t = threadIdx.x;
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
        const int64_t a = row_start[r], e = row_end[r];      // e: the row's '\n', the last field's separator
        int64_t prev = a - 1;
        int field_base = 0;
        int64_t nnz_base = WRITE ? entry_off[r] : 0;
        for (int64_t t0 = a; t0 <= e; t0 += int64_t(PARSE_THREADS) * PARSE_BYTES) {
            const int64_t p0 = t0 + int64_t(t) * PARSE_BYTES;
            int cnt = 0;
            int64_t lastp = -1;
#pragma unroll 1
            for (int k = 0; k < PARSE_BYTES; ++k) {
                const int64_t p = p0 + k;
                if (p <= e && (text[p] == ',' || text[p] == '\n') && parity[p] == 0) { ++cnt; lastp = p; }
            }
            int fbase, ftotal;
            ScanI(s_si).ExclusiveSum(cnt, fbase, ftotal);
            int64_t before, last_in_tile;
            ScanL(s_sl).ExclusiveScan(lastp, before, prev, MaxOp(), last_in_tile);
            __syncthreads();
            // pass over my separators: parse, count (and place) the nonzeros
            int my_nnz = 0;
#pragma unroll 1
            for (int pass = 0; pass < (WRITE ? 2 : 1); ++pass) {
                int64_t pos = 0;
                if (pass == 1) {
                    int excl, tot;
                    ScanI(s_si).ExclusiveSum(my_nnz, excl, tot);
                    pos = nnz_base + excl;
                    nnz_base += tot;
                }
                int f = field_base + fbase;
                int64_t q = before;
#pragma unroll 1
                for (int k = 0; k < PARSE_BYTES; ++k) {
                    const int64_t p = p0 + k;
                    if (!(p <= e && (text[p] == ',' || text[p] == '\n') && parity[p] == 0)) continue;
                    const int rl = f < nfields ? role[f] : -4;
                    if (rl == -1) {
                        if (pass == 0 && !WRITE) { lab_start[r] = q + 1; lab_end[r] = p; }
                    } else if (rl != -4) {
                        int64_t v;
                        if (!parse_count(text + q + 1, p - q - 1, &v)) {
                            if (pass == 0) atomicMin(error, ((unsigned long long)r << 32) | (unsigned)f);
                        } else if (rl == -2) {
                            if (!WRITE) seq[r] = v;
                        } else if (rl == -3) {
                            if (!WRITE) kc[r] = v;
                        } else if (v != 0) {
                            if (pass == 0) ++my_nnz;
                            else { cols[pos] = rl; vals[pos] = v; ++pos; }
                        }
                    }
                    ++f;
                    q = p;
                }
            }
            if (!WRITE) {
                int tot;
                ScanI(s_si).ExclusiveSum(my_nnz, cnt, tot);
                nnz_base += tot;
            }
            if (last_in_tile > prev) prev = last_in_tile;
            field_base += ftotal;
            __syncthreads();
        }
        if (t == 0) {
            if (field_base != nfields) atomicMin(error, ((unsigned long long)r << 32) | PARSE_FIELD_COUNT);
            if (!WRITE) row_nnz[r] = nnz_base;
        }
    }
}

inline size_t parse_rows_temp(int64_t nbytes) {
    size_t a = 0, b = 0;
    const int64_t n = nbytes > 0 ? nbytes : 1;
    cub::TransformInputIterator<uint8_t, IsQuote, const uint8_t *> q((const uint8_t *)nullptr, IsQuote());
    cub::DeviceScan::InclusiveScan(nullptr, a, q, (uint8_t *)nullptr, XorOp(), n);
    cub::DeviceSelect::If(nullptr, b, cub::CountingInputIterator<int64_t>(0), (int64_t *)nullptr, (int64_t *)nullptr, n,
                          RowEnd{nullptr, nullptr});
    return align256(a > b ? a : b);
}

}  // namespace skm

extern "C" {

int skm_csv_f64_host(double v, char *out) { return skm::fmt_f64(v, reinterpret_cast<uint8_t *>(out)); }

size_t skm_csv_rows_workspace(int64_t rows) { return skm::rows_workspace(rows); }

int skm_csv_assoc_measure(const double *d_scores, int64_t rows, int64_t A, int64_t ld, const uint8_t *d_labels,
                          const int64_t *d_label_offsets, int64_t *d_row_offsets, void *workspace, size_t workspace_bytes,
                          skm_stream_t stream) {
    using namespace skm;
    if (rows > 0 && A > 0 && (!d_scores || ld < A)) { set_error("skm_csv_assoc_measure: d_scores NULL or ld < A"); return SKM_ERR_INVALID; }
    return assoc_measure("skm_csv_assoc_measure", FullCells{d_scores, ld}, rows, A, d_labels, d_label_offsets, d_row_offsets, workspace,
                         workspace_bytes, (cudaStream_t)stream);
}

int skm_csv_assoc_write(const double *d_scores, int64_t rows, int64_t A, int64_t ld, const uint8_t *d_labels,
                        const int64_t *d_label_offsets, const int64_t *d_row_offsets, uint8_t *d_text, skm_stream_t stream) {
    using namespace skm;
    if (rows > 0 && A > 0 && (!d_scores || ld < A)) { set_error("skm_csv_assoc_write: d_scores NULL or ld < A"); return SKM_ERR_INVALID; }
    return assoc_write("skm_csv_assoc_write", FullCells{d_scores, ld}, rows, A, d_labels, d_label_offsets, d_row_offsets, d_text,
                       (cudaStream_t)stream);
}

int skm_csv_top2_measure(const int32_t *d_top1, const int32_t *d_top2, const double *d_score1, const double *d_score2, int64_t rows,
                         int64_t A, const uint8_t *d_labels, const int64_t *d_label_offsets, int64_t *d_row_offsets, void *workspace,
                         size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (rows > 0 && (!d_top1 || !d_top2 || !d_score1 || !d_score2)) { set_error("skm_csv_top2_measure: NULL argument"); return SKM_ERR_INVALID; }
    return assoc_measure("skm_csv_top2_measure", Top2Cells{d_top1, d_top2, d_score1, d_score2}, rows, A, d_labels, d_label_offsets,
                         d_row_offsets, workspace, workspace_bytes, (cudaStream_t)stream);
}

int skm_csv_top2_write(const int32_t *d_top1, const int32_t *d_top2, const double *d_score1, const double *d_score2, int64_t rows,
                       int64_t A, const uint8_t *d_labels, const int64_t *d_label_offsets, const int64_t *d_row_offsets, uint8_t *d_text,
                       skm_stream_t stream) {
    using namespace skm;
    if (rows > 0 && (!d_top1 || !d_top2 || !d_score1 || !d_score2)) { set_error("skm_csv_top2_write: NULL argument"); return SKM_ERR_INVALID; }
    return assoc_write("skm_csv_top2_write", Top2Cells{d_top1, d_top2, d_score1, d_score2}, rows, A, d_labels, d_label_offsets,
                       d_row_offsets, d_text, (cudaStream_t)stream);
}

int skm_csv_counts_measure(const int64_t *d_rowptr, const int64_t *d_vals, int64_t rows, int64_t K, const int64_t *d_seq_count,
                           const int64_t *d_kmer_count, const uint8_t *d_labels, const int64_t *d_label_offsets, int layout,
                           int64_t *d_row_offsets, void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (rows < 0 || K < 0 || (layout != 0 && layout != 1) || !d_row_offsets) { set_error("skm_csv_counts_measure: bad sizes or layout"); return SKM_ERR_INVALID; }
    int rc = check_rows_ws("skm_csv_counts_measure", rows, workspace, workspace_bytes);
    if (rc) return rc;
    if (rows > 0) {
        if (!d_rowptr || !d_seq_count || !d_kmer_count || !d_label_offsets) { set_error("skm_csv_counts_measure: NULL argument"); return SKM_ERR_INVALID; }
        counts_measure_kernel<<<grid_for(rows, CSV_WARPS), CSV_WARPS * 32, 0, (cudaStream_t)stream>>>(
            d_rowptr, d_vals, rows, K, d_seq_count, d_kmer_count, d_labels, d_label_offsets, layout, (int64_t *)workspace);
        SKM_LAUNCH_CHECK("counts_measure_kernel");
    }
    return scan_rows((int64_t *)workspace, rows, d_row_offsets, workspace, workspace_bytes, (cudaStream_t)stream);
}

int skm_csv_counts_write(const int64_t *d_rowptr, const int32_t *d_cols, const int64_t *d_vals, int64_t rows, int64_t K,
                         const int64_t *d_seq_count, const int64_t *d_kmer_count, const uint8_t *d_labels, const int64_t *d_label_offsets,
                         int layout, const int64_t *d_row_offsets, uint8_t *d_text, skm_stream_t stream) {
    using namespace skm;
    if (rows < 0 || K < 0 || (layout != 0 && layout != 1)) { set_error("skm_csv_counts_write: bad sizes or layout"); return SKM_ERR_INVALID; }
    if (rows == 0) return SKM_OK;
    if (!d_rowptr || !d_seq_count || !d_kmer_count || !d_label_offsets || !d_row_offsets || !d_text) {
        set_error("skm_csv_counts_write: NULL argument");
        return SKM_ERR_INVALID;
    }
    const int grid = (int)std::min<int64_t>(rows, int64_t(sm_count()) * 8);
    counts_write_kernel<<<grid, CNT_THREADS, 0, (cudaStream_t)stream>>>(d_rowptr, d_cols, d_vals, rows, K, d_seq_count, d_kmer_count, d_labels,
                                                                        d_label_offsets, layout, d_row_offsets, d_text);
    SKM_LAUNCH_CHECK("counts_write_kernel");
    return SKM_OK;
}

size_t skm_csv_parse_workspace(int64_t nbytes) { return skm::parse_rows_temp(nbytes); }

int skm_csv_parse_rows(const uint8_t *d_text, int64_t nbytes, uint8_t *d_parity, int64_t *d_row_ends, int64_t *d_nrows,
                       void *workspace, size_t workspace_bytes, skm_stream_t stream) {
    using namespace skm;
    if (nbytes < 0 || !d_nrows) { set_error("skm_csv_parse_rows: bad size or NULL d_nrows"); return SKM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    if (nbytes == 0) { SKM_CUDA_TRY(cudaMemsetAsync(d_nrows, 0, sizeof(int64_t), st)); return SKM_OK; }
    if (!d_text || !d_parity || !d_row_ends) { set_error("skm_csv_parse_rows: NULL argument"); return SKM_ERR_INVALID; }
    size_t need = parse_rows_temp(nbytes);
    if (!workspace || workspace_bytes < need) { set_error("skm_csv_parse_rows: workspace of %zu bytes, %zu needed", workspace_bytes, need); return SKM_ERR_WORKSPACE; }
    size_t temp = workspace_bytes;
    cub::TransformInputIterator<uint8_t, IsQuote, const uint8_t *> q(d_text, IsQuote());
    SKM_CUDA_TRY(cub::DeviceScan::InclusiveScan(workspace, temp, q, d_parity, XorOp(), nbytes, st));
    temp = workspace_bytes;
    SKM_CUDA_TRY(cub::DeviceSelect::If(workspace, temp, cub::CountingInputIterator<int64_t>(0), d_row_ends, d_nrows, nbytes,
                                       RowEnd{d_text, d_parity}, st));
    return SKM_OK;
}

int skm_csv_parse_cells(const uint8_t *d_text, const uint8_t *d_parity, const int64_t *d_row_start, const int64_t *d_row_end, int64_t rows,
                        const int32_t *d_role, int nfields, const int64_t *d_entry_offsets, int64_t *d_row_nnz, int64_t *d_seq_count,
                        int64_t *d_kmer_count, int64_t *d_label_start, int64_t *d_label_end, int32_t *d_cols, int64_t *d_vals,
                        unsigned long long *d_error, skm_stream_t stream) {
    using namespace skm;
    if (rows < 0 || nfields < 1 || rows >= (1ll << 31)) { set_error("skm_csv_parse_cells: bad sizes"); return SKM_ERR_INVALID; }
    if (rows == 0) return SKM_OK;
    if (!d_text || !d_parity || !d_row_start || !d_row_end || !d_role || !d_error) { set_error("skm_csv_parse_cells: NULL argument"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>(rows, int64_t(sm_count()) * 8);
    cudaStream_t st = (cudaStream_t)stream;
    if (!d_entry_offsets) {
        if (!d_row_nnz || !d_seq_count || !d_kmer_count || !d_label_start || !d_label_end) { set_error("skm_csv_parse_cells: NULL output"); return SKM_ERR_INVALID; }
        parse_cells_kernel<false><<<grid, PARSE_THREADS, 0, st>>>(d_text, d_parity, d_row_start, d_row_end, rows, d_role, nfields, nullptr, d_row_nnz,
                                                                  d_seq_count, d_kmer_count, d_label_start, d_label_end, nullptr, nullptr, d_error);
    } else {
        if (!d_cols || !d_vals) { set_error("skm_csv_parse_cells: NULL d_cols / d_vals"); return SKM_ERR_INVALID; }
        parse_cells_kernel<true><<<grid, PARSE_THREADS, 0, st>>>(d_text, d_parity, d_row_start, d_row_end, rows, d_role, nfields, d_entry_offsets,
                                                                 nullptr, nullptr, nullptr, nullptr, nullptr, d_cols, d_vals, d_error);
    }
    SKM_LAUNCH_CHECK("parse_cells_kernel");
    return SKM_OK;
}

}  // extern "C"
