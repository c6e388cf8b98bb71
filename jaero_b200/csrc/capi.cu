// extern "C" boundary of libjaero_b200.so (declared in include/jaero_b200.h): error state, the device lifecycle helpers of
// handle.cuh, and the Viterbi handle. The other handle families are in capi_batch.cu (demodulator batches), capi_burst.cu
// (burst demodulators), capi_frames.cu (P, C and R/T frame layers), capi_ingest.cu (ingest router) and channelizer.cu.
// Host-side object management only: device allocation, staging copies, stream ordering, kernel launches. No CPU
// implementation of any DSP lives here — without a CUDA device every create call fails loudly.
#include "capi_internal.cuh"
#include "viterbi.cuh"
#include <algorithm>
#include <cstring>

namespace jb {
static thread_local std::string g_err;
void set_error(const std::string &m) { g_err = m; }
int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d in %s", (int)e, cudaGetErrorString(e), file, line, what);
    g_err = buf;
    return JAERO_E_CUDA;
}
int open_device(int device, const char *who)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); n = 0; }
    if (device < 0 || device >= n) { set_error(std::string(who) + ": no such CUDA device (there is no CPU fallback)"); return JAERO_E_CUDA; }
    JB_CUDA(cudaSetDevice(device));
    return JAERO_OK;
}
int read_soft_rows(const int *cnt, const int *ovf, int C, const int16_t *d_soft, int soft_cap, int16_t *h_stage, int16_t *out,
                   size_t cap, int32_t *counts, cudaStream_t s)
{
    int maxc = 0; bool overflow = false;
    for (int ch = 0; ch < C; ch++) { maxc = std::max(maxc, cnt[ch]); overflow |= (ovf[ch] != 0) || ((size_t)cnt[ch] > cap); }
    if (overflow) { set_error("soft-bit ring overflow: drain more often or pass a larger buffer"); return JAERO_E_OVERFLOW; }
    if (maxc > 0) {
        JB_CUDA(cudaMemcpy2DAsync(h_stage, (size_t)soft_cap * 2, d_soft, (size_t)soft_cap * 2, (size_t)maxc * 2, C, cudaMemcpyDeviceToHost, s));
        JB_CUDA(cudaStreamSynchronize(s));
    }
    for (int ch = 0; ch < C; ch++) {
        counts[ch] = cnt[ch];
        if (cnt[ch]) memcpy(out + (size_t)ch * cap, h_stage + (size_t)ch * soft_cap, (size_t)cnt[ch] * 2);
    }
    return JAERO_OK;
}
} // namespace jb
using namespace jb;

struct jaero_viterbi {
    int device; cudaStream_t stream;
    HandleAllocs allocs;
    int n_channels, pad;
    uint8_t *d_overlap; int *d_overlap_len; int *d_renorm;
    GrowBuffer<uint8_t> soft, bits;
    int *d_valid;
    int64_t launches;
};

extern "C" {

const char *jaero_last_error(void) { return g_err.c_str(); }
int jaero_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ------------------------------------------------------------------ Viterbi
int jaero_viterbi_create(int n_channels, int paddinglength, int device, jaero_viterbi **out)
{
    if (!out || n_channels <= 0 || paddinglength < 0 || (paddinglength & 1)) { set_error("jaero_viterbi_create: bad argument"); return JAERO_E_ARG; }
    NewHandle<jaero_viterbi> nh(jaero_viterbi_destroy);
    int r = nh.open(device, "jaero_viterbi_create"); if (r) return r;
    jaero_viterbi *v = nh.h;
    v->n_channels = n_channels; v->pad = paddinglength;
    const size_t C = n_channels;
    if (v->allocs.zeroed(&v->d_overlap, C * 64, v->stream) || v->allocs.zeroed(&v->d_overlap_len, C, v->stream) ||
        v->allocs.zeroed(&v->d_renorm, C, v->stream) || v->allocs.zeroed(&v->d_valid, C, v->stream)) return JAERO_E_CUDA;
    *out = nh.release();
    return JAERO_OK;
}
void jaero_viterbi_destroy(jaero_viterbi *v)
{
    if (!v) return;
    cudaSetDevice(v->device);
    cudaStreamSynchronize(v->stream);
    v->allocs.free_all(); v->soft.release(); v->bits.release();
    cudaStreamDestroy(v->stream);
    delete v;
}
int jaero_viterbi_reset(jaero_viterbi *v)
{
    if (!v) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(v->device));
    JB_CUDA(cudaMemsetAsync(v->d_overlap_len, 0, (size_t)v->n_channels * sizeof(int), v->stream));
    return JAERO_OK;
}
int jaero_viterbi_sync(jaero_viterbi *v)
{
    if (!v) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(v->device));
    JB_CUDA(cudaStreamSynchronize(v->stream));
    return JAERO_OK;
}
int64_t jaero_viterbi_launch_count(const jaero_viterbi *v) { return v ? v->launches : 0; }

static int vit_check(jaero_viterbi *v, size_t n_soft, int cols)
{
    if (!v) { set_error("null handle"); return JAERO_E_ARG; }
    if (n_soft < 32 || (n_soft & 1) || n_soft > 60000) { set_error("viterbi: n_soft must be even, 32..60000"); return JAERO_E_ARG; }
    if (cols < 0 || (cols > 0 && (size_t)cols * 64 != n_soft)) { set_error("viterbi: interleaver_cols*64 must equal n_soft"); return JAERO_E_ARG; }
    return JAERO_OK;
}
int jaero_viterbi_decode_continuous_device(jaero_viterbi *v, const uint8_t *d_soft, size_t n_soft, int cols, uint8_t *d_bits, int32_t *d_n_valid)
{
    int r = vit_check(v, n_soft, cols); if (r) return r;
    JB_CUDA(cudaSetDevice(v->device));
    if (viterbi_launch(d_soft, (int)n_soft, cols, 0, v->pad, v->d_overlap, v->d_overlap_len, v->d_renorm, d_bits, d_n_valid, v->n_channels, v->stream)) return JAERO_E_CUDA;
    v->launches++;
    return JAERO_OK;
}
// host soft values in, staged on the device: the decoded bits land in v->bits
static int vit_stage(jaero_viterbi *v, const uint8_t *soft, size_t n_soft)
{
    const size_t C = v->n_channels;
    if (v->soft.reserve(C * n_soft, v->stream) || v->bits.reserve(C * (n_soft / 2), v->stream)) return JAERO_E_CUDA;
    JB_CUDA(cudaMemcpyAsync(v->soft.ptr, soft, C * n_soft, cudaMemcpyHostToDevice, v->stream));
    return JAERO_OK;
}
int jaero_viterbi_decode_continuous(jaero_viterbi *v, const uint8_t *soft, size_t n_soft, int cols, uint8_t *bits_out, int32_t *n_valid)
{
    int r = vit_check(v, n_soft, cols); if (r) return r;
    if (!soft || !bits_out) { set_error("null buffer"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(v->device));
    r = vit_stage(v, soft, n_soft); if (r) return r;
    r = jaero_viterbi_decode_continuous_device(v, v->soft.ptr, n_soft, cols, v->bits.ptr, v->d_valid); if (r) return r;
    JB_CUDA(cudaMemcpyAsync(bits_out, v->bits.ptr, (size_t)v->n_channels * (n_soft / 2), cudaMemcpyDeviceToHost, v->stream));
    if (n_valid) JB_CUDA(cudaMemcpyAsync(n_valid, v->d_valid, (size_t)v->n_channels * sizeof(int), cudaMemcpyDeviceToHost, v->stream));
    JB_CUDA(cudaStreamSynchronize(v->stream));
    return JAERO_OK;
}
int jaero_viterbi_decode_block(jaero_viterbi *v, const uint8_t *soft, size_t n_soft, uint8_t *bits_out)
{
    int r = vit_check(v, n_soft, 0); if (r) return r;
    if (!soft || !bits_out) { set_error("null buffer"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(v->device));
    r = vit_stage(v, soft, n_soft); if (r) return r;
    if (viterbi_launch(v->soft.ptr, (int)n_soft, 0, 1, 0, v->d_overlap, v->d_overlap_len, v->d_renorm, v->bits.ptr, v->d_valid, v->n_channels, v->stream)) return JAERO_E_CUDA;
    v->launches++;
    JB_CUDA(cudaMemcpyAsync(bits_out, v->bits.ptr, (size_t)v->n_channels * (n_soft / 2), cudaMemcpyDeviceToHost, v->stream));
    JB_CUDA(cudaStreamSynchronize(v->stream));
    return JAERO_OK;
}

} // extern "C"
