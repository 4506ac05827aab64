// skm_confidence.cu — the device side of the confidence evaluation (rule `evaluate`, class Evaluator,
// learn.smk:923-1348) and of reading score matrices back (learn.smk:964-981).
//
//  skm_top2_rows_f64     per row of a float64 score matrix with NaN holes (the top-2-masked
//                        seq-annotation-scores CSV): column of the maximum (NaN skipped, first maximum — idxmax)
//                        and the two largest values (argpartition(-values, [0, 1]): NaN last).
//  skm_confidence_hist   Difference bin of every query, -(round(Second - Top, 2)) * 100 as numpy computes it
//                        (rint(x * 100) / 100), and the per-(prediction, bin) counts of the Known rows, True and
//                        False predictions separately (pd.crosstab, learn.smk:1052-1061).  The T / F / skip
//                        class of a row is an input: the reference decides it with substring tests on the row
//                        label (learn.smk:997-1008).
//  skm_confidence_classify  that class for the rows of eval_apply (learn.smk:712-732), whose label is
//                        `<annotation>_known_<n>` or `<accession>_unknown_<n>`: the substring tests run on the name
//                        table and the row number, so the label strings never exist.
// Integer atomics only: the histograms are order-independent, hence reproducible.
#include "skm_common.cuh"

namespace skm {

struct Top2v {
    double s1, s2;
    int i1, i2;
};
// larger value first; equal values -> lower column (first maximum)
__device__ __forceinline__ void top2v_push(Top2v &t, double s, int i) {
    if (i < 0) return;
    if (t.i1 < 0 || s > t.s1 || (s == t.s1 && i < t.i1)) { t.s2 = t.s1; t.i2 = t.i1; t.s1 = s; t.i1 = i; }
    else if (t.i2 < 0 || s > t.s2 || (s == t.s2 && i < t.i2)) { t.s2 = s; t.i2 = i; }
}

__global__ void __launch_bounds__(256) top2_rows_f64_kernel(const double *__restrict__ S, int64_t nq, int64_t A,
                                                            int32_t *__restrict__ top1, int32_t *__restrict__ top2,
                                                            double *__restrict__ s1, double *__restrict__ s2) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    for (int64_t q = warp; q < nq; q += nwarps) {
        const double *row = S + q * A;
        Top2v t{0.0, 0.0, -1, -1};
        for (int64_t a = lane; a < A; a += 32) {
            const double v = row[a];
            if (v == v) top2v_push(t, v, int(a));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double os1 = __shfl_xor_sync(FULL, t.s1, o), os2 = __shfl_xor_sync(FULL, t.s2, o);
            const int oi1 = __shfl_xor_sync(FULL, t.i1, o), oi2 = __shfl_xor_sync(FULL, t.i2, o);
            top2v_push(t, os1, oi1);
            top2v_push(t, os2, oi2);
        }
        if (lane == 0) {
            top1[q] = t.i1; top2[q] = t.i2;
            s1[q] = t.i1 >= 0 ? t.s1 : nan("");
            s2[q] = t.i2 >= 0 ? t.s2 : nan("");
        }
    }
}

constexpr int CONF_BINS = 101;

// cls[q]: 0 = not counted (Unknown row), 1 = Known & True, 2 = Known & False
__global__ void __launch_bounds__(256) confidence_hist_kernel(const int32_t *__restrict__ top1, const double *__restrict__ s1,
                                                              const double *__restrict__ s2, const uint8_t *__restrict__ cls,
                                                              int64_t nq, int64_t n_ann, unsigned long long *__restrict__ hist_t,
                                                              unsigned long long *__restrict__ hist_f, uint8_t *__restrict__ bin_out) {
    for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q < nq; q += int64_t(gridDim.x) * blockDim.x) {
        const int p = top1[q];
        // numpy: round(x, 2) = rint(x * 100) / 100; Difference = -(that).  No FMA contraction: a lone product.
        const double t = rint(__dmul_rn(__dsub_rn(s2[q], s1[q]), 100.0));
        int bin = 255;
        if (p >= 0 && p < n_ann && t == t && t <= 0.0 && t >= -100.0) bin = int(-t);
        if (bin_out) bin_out[q] = uint8_t(bin);
        if (bin == 255 || !cls) continue;
        const uint8_t c = cls[q];
        if (c == 1) atomicAdd(hist_t + int64_t(p) * CONF_BINS + bin, 1ull);
        else if (c == 2) atomicAdd(hist_f + int64_t(p) * CONF_BINS + bin, 1ull);
    }
}

// "_known_" + decimal(v) (v < 2^63: at most 7 + 19 bytes), little-endian in four registers: a local array indexed by
// a run-time position would live in local memory.
struct KnownSuffix {
    uint64_t w0, w1, w2, w3;
    int len;
};

__host__ __device__ __forceinline__ KnownSuffix known_suffix(uint64_t v) {
    int nd = 1;
    for (uint64_t t = v; t >= 10; t /= 10) ++nd;
    KnownSuffix s{0x005f6e776f6e6b5full, 0, 0, 0, 7 + nd};     // "_known_"
#pragma unroll
    for (int i = 0; i < 20; ++i) {
        if (i < nd) {
            const int pos = 7 + nd - 1 - i;
            const uint64_t b = uint64_t('0' + int(v % 10)) << ((pos & 7) * 8);
            const int w = pos >> 3;
            s.w0 |= w == 0 ? b : 0;
            s.w1 |= w == 1 ? b : 0;
            s.w2 |= w == 2 ? b : 0;
            s.w3 |= w == 3 ? b : 0;
            v /= 10;
        }
    }
    return s;
}

__host__ __device__ __forceinline__ uint8_t suffix_byte(const KnownSuffix &s, int64_t j) {
    const uint64_t w = j < 8 ? s.w0 : j < 16 ? s.w1 : j < 24 ? s.w2 : s.w3;
    return uint8_t(w >> ((j & 7) * 8));
}

// Python `needle in name + suffix` on UTF-8 bytes (byte substring == code-point substring for valid UTF-8); the
// empty needle is in everything.  Plain search: names are short, and a row stops at its first match.
__host__ __device__ __forceinline__ bool label_contains(const uint8_t *__restrict__ needle, int64_t m,
                                                        const uint8_t *__restrict__ name, int64_t nt, const KnownSuffix &sfx) {
    const int64_t L = nt + sfx.len;
    if (m > L) return false;
    for (int64_t st = 0; st + m <= L; ++st) {
        int64_t j = 0;
        for (; j < m; ++j) {
            const int64_t h = st + j;
            if (needle[j] != (h < nt ? name[h] : suffix_byte(sfx, h - nt))) break;
        }
        if (j == m) return true;
    }
    return false;
}

__host__ __device__ __forceinline__ bool contains_unknown(const uint8_t *__restrict__ name, int64_t n) {
    constexpr uint64_t UNKNOWN = 0x006e776f6e6b6e75ull;          // "unknown"
    for (int64_t st = 0; st + 7 <= n; ++st) {
        int j = 0;
        for (; j < 7; ++j)
            if (name[st + j] != uint8_t(UNKNOWN >> (8 * j))) break;
        if (j == 7) return true;
    }
    return false;
}

// Class of row q (learn.smk:997-1008): 0 Unknown, 1 Known & True, 2 Known & False.  The label of an unknown row
// contains "unknown"; a known label contains it only through its annotation name, since "_known_<digits>" cannot
// complete it.  An index outside [0, n_names) is no name: truth -> Unknown, top1 -> False.
__host__ __device__ __forceinline__ uint8_t classify_row(int32_t p, int32_t t, uint64_t row, const uint8_t *__restrict__ names,
                                                         const int64_t *__restrict__ off, int64_t n_names) {
    if (t < 0 || t >= n_names) return 0;
    const uint8_t *name = names + off[t];
    const int64_t nt = off[t + 1] - off[t];
    if (contains_unknown(name, nt)) return 0;
    if (p == t) return 1;
    if (p < 0 || p >= n_names) return 2;
    return label_contains(names + off[p], off[p + 1] - off[p], name, nt, known_suffix(row)) ? 1 : 2;
}

__global__ void __launch_bounds__(256) confidence_classify_kernel(const int32_t *__restrict__ top1, const int32_t *__restrict__ truth,
                                                                  int64_t nq, int64_t row_base, const uint8_t *__restrict__ names,
                                                                  const int64_t *__restrict__ off, int64_t n_names,
                                                                  uint8_t *__restrict__ cls) {
    for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q < nq; q += int64_t(gridDim.x) * blockDim.x)
        cls[q] = classify_row(top1[q], truth[q], uint64_t(row_base + q), names, off, n_names);
}

}  // namespace skm

extern "C" {

int skm_top2_rows_f64(const double *d_scores, int64_t nq, int64_t n_ann, int32_t *d_top1, int32_t *d_top2,
                      double *d_score1, double *d_score2, skm_stream_t stream) {
    using namespace skm;
    if (nq < 0 || n_ann < 0 || n_ann >= (1ll << 31)) { set_error("skm_top2_rows_f64: bad sizes"); return SKM_ERR_INVALID; }
    if (nq == 0) return SKM_OK;
    if ((n_ann > 0 && !d_scores) || !d_top1 || !d_top2 || !d_score1 || !d_score2) { set_error("skm_top2_rows_f64: NULL argument"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>((nq + 7) / 8, int64_t(sm_count()) * 8);
    top2_rows_f64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_scores, nq, n_ann, d_top1, d_top2, d_score1, d_score2);
    SKM_LAUNCH_CHECK("top2_rows_f64_kernel");
    return SKM_OK;
}

int skm_confidence_hist(const int32_t *d_top1, const double *d_score1, const double *d_score2, const uint8_t *d_class,
                        int64_t nq, int64_t n_ann, int64_t *d_hist_true, int64_t *d_hist_false, uint8_t *d_bin_out,
                        skm_stream_t stream) {
    using namespace skm;
    if (nq < 0 || n_ann < 0) { set_error("skm_confidence_hist: negative size"); return SKM_ERR_INVALID; }
    if (nq == 0) return SKM_OK;
    if (!d_top1 || !d_score1 || !d_score2) { set_error("skm_confidence_hist: NULL argument"); return SKM_ERR_INVALID; }
    if (d_class && (!d_hist_true || !d_hist_false)) { set_error("skm_confidence_hist: classes given without histograms"); return SKM_ERR_INVALID; }
    if (!d_class && !d_bin_out) { set_error("skm_confidence_hist: nothing to compute"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>((nq + 255) / 256, int64_t(sm_count()) * 8);
    confidence_hist_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_top1, d_score1, d_score2, d_class, nq, n_ann,
                                                                   reinterpret_cast<unsigned long long *>(d_hist_true),
                                                                   reinterpret_cast<unsigned long long *>(d_hist_false), d_bin_out);
    SKM_LAUNCH_CHECK("confidence_hist_kernel");
    return SKM_OK;
}

int skm_confidence_classify(const int32_t *d_top1, const int32_t *d_truth, int64_t nq, int64_t row_base,
                            const uint8_t *d_names, const int64_t *d_name_offsets, int64_t n_names, uint8_t *d_class,
                            skm_stream_t stream) {
    using namespace skm;
    if (nq < 0 || n_names < 0 || n_names >= (1ll << 31)) { set_error("skm_confidence_classify: bad sizes"); return SKM_ERR_INVALID; }
    if (row_base < 0 || row_base > INT64_MAX - nq) { set_error("skm_confidence_classify: row numbers outside [0, 2^63)"); return SKM_ERR_INVALID; }
    if (nq == 0) return SKM_OK;
    if (!d_top1 || !d_truth || !d_class || (n_names > 0 && !d_name_offsets)) { set_error("skm_confidence_classify: NULL argument"); return SKM_ERR_INVALID; }
    const int grid = (int)std::min<int64_t>((nq + 255) / 256, int64_t(sm_count()) * 8);
    confidence_classify_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_top1, d_truth, nq, row_base, d_names, d_name_offsets,
                                                                       n_names, d_class);
    SKM_LAUNCH_CHECK("confidence_classify_kernel");
    return SKM_OK;
}

}  // extern "C"
