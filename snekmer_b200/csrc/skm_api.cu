// skm_api.cu — error plumbing, device query, host-side LUT builder, argument checks.
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "skm_common.cuh"

namespace skm {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return SKM_ERR_CUDA;
}

int sm_count() {
    static thread_local int cached = 0, cached_dev = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

int check_common(const void *d_residues, int64_t nres, const void *d_offsets, int64_t nseq,
                 const void *d_lut, int nsym, int k) {
    if (nres < 0 || nseq < 0) { set_error("negative size (nres=%lld nseq=%lld)", (long long)nres, (long long)nseq); return SKM_ERR_INVALID; }
    if (nseq > 0 && !d_offsets) { set_error("d_offsets is NULL"); return SKM_ERR_INVALID; }
    if (nres > 0 && !d_residues) { set_error("d_residues is NULL"); return SKM_ERR_INVALID; }
    if ((reinterpret_cast<uintptr_t>(d_residues) & 15u) != 0) { set_error("d_residues must be 16-byte aligned"); return SKM_ERR_INVALID; }
    if (!d_lut) { set_error("d_lut is NULL"); return SKM_ERR_INVALID; }
    if (nsym < 1 || nsym > 254) { set_error("nsym=%d out of range [1,254]", nsym); return SKM_ERR_INVALID; }
    if (k < 1 || k > SKM_MAX_K) { set_error("k=%d out of range [1,%d]", k, SKM_MAX_K); return SKM_ERR_INVALID; }
    unsigned __int128 s;
    if (!code_space(nsym, k, &s)) { set_error("nsym^k = %d^%d does not fit 64-bit codes", nsym, k); return SKM_ERR_UNSUPPORTED; }
    return SKM_OK;
}

}  // namespace skm

extern "C" {

int skm_version(void) { return 20400; /* 2.4.0 */ }

const char *skm_last_error(void) { return skm::g_err; }

int skm_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    SKM_CUDA_TRY(cudaGetDevice(&dev));
    int n = 0, ma = 0, mi = 0;
    SKM_CUDA_TRY(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    SKM_CUDA_TRY(cudaDeviceGetAttribute(&ma, cudaDevAttrComputeCapabilityMajor, dev));
    SKM_CUDA_TRY(cudaDeviceGetAttribute(&mi, cudaDevAttrComputeCapabilityMinor, dev));
    if (sm_count) *sm_count = n;
    if (cc_major) *cc_major = ma;
    if (cc_minor) *cc_minor = mi;
    return SKM_OK;
}

int skm_lut_build(const char *map_from, const char *map_to, int nmap, const char *symbols, int nsym,
                  uint8_t lut_out[256]) {
    if (!lut_out || !symbols || nsym < 1 || nsym > 254 || nmap < 0 || (nmap > 0 && (!map_from || !map_to))) {
        skm::set_error("skm_lut_build: bad arguments");
        return SKM_ERR_INVALID;
    }
    unsigned char trans[256];
    for (int b = 0; b < 256; ++b) trans[b] = (unsigned char)b;   // str.translate: unmapped stay
    for (int i = 0; i < nmap; ++i) trans[(unsigned char)map_from[i]] = (unsigned char)map_to[i];
    int sym_index[256];
    for (int b = 0; b < 256; ++b) sym_index[b] = -1;
    for (int i = 0; i < nsym; ++i) {
        unsigned char c = (unsigned char)symbols[i];
        if (sym_index[c] >= 0) { skm::set_error("skm_lut_build: duplicate symbol '%c'", c); return SKM_ERR_INVALID; }
        sym_index[c] = i;
    }
    for (int b = 0; b < 256; ++b) {
        int s = (b < 128) ? sym_index[trans[b]] : -1;            // non-ASCII bytes are never symbols
        lut_out[b] = (s >= 0) ? (uint8_t)s : (uint8_t)SKM_INVALID_SYMBOL;
    }
    return SKM_OK;
}

}  // extern "C"
