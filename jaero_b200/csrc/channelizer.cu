// Device channelizer (include/jaero_b200.h, "device channelizer"): one wideband complex IQ stream in, one real int16 audio
// row per channel out, in the layout jaero_batch_write_device consumes.
//
// phi_c(mD - k) = phi_c(mD) - phi_c(k) holds exactly in uint32 phase arithmetic, so the mix-to-0-Hz, low-pass and decimate of
// every channel is one complex matrix product shared by all channels:
//   A[c][m] = sum_k G[c][k] X[k][m],   G[c][k] = h[k] e^{+2 pi j phi_c(k) / 2^32},   X[k][m] = x[mD - k],
// followed per output by one rotation through (psi(m) - phi_c(mD)) mod 2^32, the gain, rounding and saturation.
// G is built once at create (double, stored as float2); x is kept as float2 behind a copy of the last Tpad-1 input samples
// (shared by all channels; channels carry no other state). chan_ddc_kernel runs k in a fixed ascending order for every
// output, so each output's sum does not depend on how the input was cut into writes.
#include "../../include/jaero_b200.h"
#include "handle.cuh"
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

using namespace jb;

namespace {

constexpr int TILE_C = 64;    // channels per block
constexpr int TILE_M = 128;   // outputs per block
constexpr int KC = 16;        // taps per shared-memory chunk
constexpr int THREADS = 256;  // 16 x 16; each thread holds 4 channels x 8 outputs of complex FP32 accumulators
constexpr int RC = TILE_C / 16, RM = TILE_M / 16;

// x[n] as float2 into cur[H + i]; cur[0..H) = the last H samples of the previous write's buffer (zeros before the first write)
__global__ void chan_convert_kernel(const void *__restrict__ iq, int fmt, long long n, const float2 *__restrict__ prev,
                                    long long prev_n, int H, float2 *__restrict__ cur)
{
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= H + n) return;
    if (i < H) {
        cur[i] = prev ? prev[prev_n + i] : make_float2(0.f, 0.f);
        return;
    }
    long long s = i - H;
    float2 v;
    if (fmt == JAERO_IQ_CS16) {
        short2 q = reinterpret_cast<const short2 *>(iq)[s];
        v = make_float2((float)q.x, (float)q.y);
    } else {
        uchar2 q = reinterpret_cast<const uchar2 *>(iq)[s];
        v = make_float2((float)q.x * 256.f - 32640.f, (float)q.y * 256.f - 32640.f);   // ((u - 127.5) * 256), exact
    }
    cur[i] = v;
}

// One block: TILE_C channels x TILE_M outputs. G is [Tpad][Cpad] (tap-major, zero beyond T and C); xb[pos] with
// pos = off0 + j*D - k for local output j; out[c*stride + j].
__global__ void __launch_bounds__(THREADS) chan_ddc_kernel(const float2 *__restrict__ G, int Cpad, int Tpad, int C,
                                                           const float2 *__restrict__ xb, long long off0, int D, int M,
                                                           unsigned long long m_first, const uint32_t *__restrict__ inc_c,
                                                           uint32_t inc_a, double gain, int16_t *__restrict__ out, size_t stride)
{
    __shared__ float2 Gs[KC][TILE_C];
    __shared__ float2 Xs[KC][TILE_M + 1];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int c0 = blockIdx.y * TILE_C, j0 = blockIdx.x * TILE_M;
    float2 acc[RC][RM];
#pragma unroll
    for (int i = 0; i < RC; i++)
#pragma unroll
        for (int j = 0; j < RM; j++) acc[i][j] = make_float2(0.f, 0.f);

    for (int k0 = 0; k0 < Tpad; k0 += KC) {
#pragma unroll
        for (int r = 0; r < KC * TILE_C / THREADS; r++) {
            int e = tid + r * THREADS, kk = e / TILE_C, cc = e % TILE_C;
            Gs[kk][cc] = G[(size_t)(k0 + kk) * Cpad + c0 + cc];
        }
#pragma unroll
        for (int r = 0; r < KC * TILE_M / THREADS; r++) {
            int e = tid + r * THREADS, kk = e % KC, mm = e / KC, j = j0 + mm;
            Xs[kk][mm] = j < M ? xb[off0 + (long long)j * D - (k0 + kk)] : make_float2(0.f, 0.f);
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < KC; kk++) {
            float2 g[RC], x[RM];
#pragma unroll
            for (int i = 0; i < RC; i++) g[i] = Gs[kk][ty + 16 * i];
#pragma unroll
            for (int j = 0; j < RM; j++) x[j] = Xs[kk][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < RC; i++)
#pragma unroll
                for (int j = 0; j < RM; j++) {
                    acc[i][j].x = fmaf(g[i].x, x[j].x, acc[i][j].x);
                    acc[i][j].x = fmaf(-g[i].y, x[j].y, acc[i][j].x);
                    acc[i][j].y = fmaf(g[i].x, x[j].y, acc[i][j].y);
                    acc[i][j].y = fmaf(g[i].y, x[j].x, acc[i][j].y);
                }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < RC; i++) {
        int c = c0 + ty + 16 * i;
        if (c >= C) continue;
        uint32_t ic = inc_c[c];
#pragma unroll
        for (int j = 0; j < RM; j++) {
            int jj = j0 + tx + 16 * j;
            if (jj >= M) continue;
            unsigned long long m = m_first + jj;
            uint32_t phi = ic * (uint32_t)(m * (unsigned long long)D);   // phi_c(mD), mod 2^32
            uint32_t psi = inc_a * (uint32_t)m;
            int32_t th = (int32_t)(psi - phi);
            double s, co;
            sincospi((double)th * (1.0 / 2147483648.0), &s, &co);
            double v = gain * ((double)acc[i][j].x * co - (double)acc[i][j].y * s);
            v = rint(v);
            v = fmin(fmax(v, -32768.0), 32767.0);
            out[(size_t)c * stride + jj] = (int16_t)v;
        }
    }
}

double bessel_i0(double x)
{
    double sum = 1.0, term = 1.0, q = 0.25 * x * x;
    for (int k = 1; k < 500; k++) {
        term *= q / ((double)k * k);
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

// Validates the settings and designs h (scipy.signal.firwin(T, (f_p + f_s)/2, window=('kaiser', beta), fs=input_rate) with T
// from kaiserord(60, (f_s - f_p) / (input_rate / 2)), made odd). Returns T or JAERO_E_ARG.
int chan_design(const jaero_chan_settings *s, std::vector<double> *h, int *D_out)
{
    if (!s) { set_error("jaero_chan: null settings"); return JAERO_E_ARG; }
    if (s->iq_format != JAERO_IQ_CS16 && s->iq_format != JAERO_IQ_CU8) { set_error("jaero_chan: unknown iq_format"); return JAERO_E_ARG; }
    if (!std::isfinite(s->input_rate) || !std::isfinite(s->output_rate) || s->input_rate <= 0 || s->output_rate <= 0) {
        set_error("jaero_chan: input_rate and output_rate must be positive"); return JAERO_E_ARG; }
    double r = s->input_rate / s->output_rate;
    double Dd = std::floor(r + 0.5);
    if (std::fabs(r - Dd) > 1e-9 * r || Dd < 2 || Dd > 1e6) {
        set_error("jaero_chan: input_rate / output_rate must be an integer D >= 2"); return JAERO_E_ARG; }
    if (!std::isfinite(s->audio_hz) || s->audio_hz <= 0 || s->audio_hz >= 0.5 * s->output_rate) {
        set_error("jaero_chan: audio_hz must lie in (0, output_rate/2)"); return JAERO_E_ARG; }
    if (!std::isfinite(s->passband_hz) || s->passband_hz <= 0) { set_error("jaero_chan: passband_hz must be positive"); return JAERO_E_ARG; }
    if (!std::isfinite(s->gain) || s->gain <= 0) { set_error("jaero_chan: gain must be positive and finite"); return JAERO_E_ARG; }
    const double A = 60.0;
    double fp = 0.5 * s->passband_hz;
    double fs = std::fmin(2 * s->audio_hz, s->output_rate - 2 * s->audio_hz) - fp;
    if (!(fs > fp)) { set_error("jaero_chan: no transition band (f_s <= f_p): narrow the passband or move audio_hz"); return JAERO_E_ARG; }
    double width = (fs - fp) / (0.5 * s->input_rate);
    double numtaps = (A - 7.95) / 2.285 / (M_PI * width) + 1;
    if (!(numtaps <= JAERO_CHAN_MAX_TAPS)) { set_error("jaero_chan: filter longer than 8191 taps"); return JAERO_E_ARG; }
    int T = (int)std::ceil(numtaps);
    if (!(T & 1)) T++;
    if (T > JAERO_CHAN_MAX_TAPS) { set_error("jaero_chan: filter longer than 8191 taps"); return JAERO_E_ARG; }
    if (h) {
        const double beta = 0.1102 * (A - 8.7), cut = (fp + fs) / 2 / (0.5 * s->input_rate), alpha = 0.5 * (T - 1);
        const double i0b = bessel_i0(beta);
        h->assign(T, 0.0);
        double sum = 0;
        for (int n = 0; n < T; n++) {
            double m = n - alpha, xm = cut * m;
            double sinc = xm == 0 ? 1.0 : std::sin(M_PI * xm) / (M_PI * xm);
            double u = (n - alpha) / alpha;
            double w = bessel_i0(beta * std::sqrt(1 - u * u)) / i0b;
            (*h)[n] = cut * sinc * w;
            sum += (*h)[n];
        }
        for (int n = 0; n < T; n++) (*h)[n] /= sum;
    }
    if (D_out) *D_out = (int)Dd;
    return T;
}

} // namespace

struct jaero_chan {
    int device, C, Cpad, T, Tpad, H, D, fmt;
    double gain;
    uint32_t inc_a;
    cudaStream_t stream, own_stream;
    HandleAllocs allocs;
    float2 *d_G;
    uint32_t *d_inc;
    GrowBuffer<float2> x[2]; int cur; long long last_n;            // ping-pong sample buffers, H history + last write
    bool have_prev;
    GrowBuffer<uint8_t> raw;                                        // staging for host writes
    GrowBuffer<int16_t> out; size_t stride, n_out;                  // [C][stride]
    long long n_in;                                                 // input samples so far
    int64_t launches;
};

extern "C" {

int jaero_chan_taps(const jaero_chan_settings *s, double *taps, int cap)
{
    std::vector<double> h;
    int T = chan_design(s, taps ? &h : nullptr, nullptr);
    if (T < 0) return T;
    if (taps)
        for (int k = 0; k < T && k < cap; k++) taps[k] = h[k];
    return T;
}

void jaero_chan_destroy(jaero_chan *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    c->allocs.free_all(); c->x[0].release(); c->x[1].release(); c->raw.release(); c->out.release();
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

int jaero_chan_create(const jaero_chan_settings *s, int n_channels, const double *offset_hz, int device, jaero_chan **out)
{
    if (!out || n_channels <= 0 || !offset_hz) { set_error("jaero_chan_create: bad argument (n_channels must be positive)"); return JAERO_E_ARG; }
    std::vector<double> h;
    int D = 0;
    int T = chan_design(s, &h, &D);
    if (T < 0) return T;
    for (int c = 0; c < n_channels; c++) {
        double o = offset_hz[c];
        if (!std::isfinite(o) || std::fabs(o) + 0.5 * s->passband_hz > 0.5 * s->input_rate) {
            set_error("jaero_chan_create: channel " + std::to_string(c) + " does not fit inside the input band"); return JAERO_E_ARG; }
    }
    NewHandle<jaero_chan> nh(jaero_chan_destroy);
    int r = nh.open(device, "jaero_chan_create"); if (r) return r;
    jaero_chan *c = nh.h;
    c->own_stream = c->stream;
    c->C = n_channels; c->T = T; c->D = D; c->fmt = s->iq_format; c->gain = s->gain;
    c->Cpad = (n_channels + TILE_C - 1) / TILE_C * TILE_C;
    c->Tpad = (T + KC - 1) / KC * KC;
    c->H = c->Tpad - 1;
    c->inc_a = (uint32_t)(int64_t)llround(s->audio_hz / s->output_rate * 4294967296.0);
    std::vector<uint32_t> inc(n_channels);
    for (int k = 0; k < n_channels; k++) inc[k] = (uint32_t)(int64_t)llround(offset_hz[k] / s->input_rate * 4294967296.0);
    std::vector<float2> G((size_t)c->Tpad * c->Cpad, make_float2(0.f, 0.f));
    for (int k = 0; k < T; k++)
        for (int ch = 0; ch < n_channels; ch++) {
            uint32_t ph = inc[ch] * (uint32_t)k;
            double a = 2.0 * M_PI * (double)ph / 4294967296.0;
            G[(size_t)k * c->Cpad + ch] = make_float2((float)(h[k] * std::cos(a)), (float)(h[k] * std::sin(a)));
        }
    if (c->allocs.upload(&c->d_G, G, c->stream) || c->allocs.upload(&c->d_inc, inc, c->stream)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(c->stream));
    *out = nh.release();
    return JAERO_OK;
}

int jaero_chan_set_stream(jaero_chan *c, void *cuda_stream)
{
    if (!c) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    JB_CUDA(cudaStreamSynchronize(c->stream));
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return JAERO_OK;
}

int jaero_chan_sync(jaero_chan *c)
{
    if (!c) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    JB_CUDA(cudaStreamSynchronize(c->stream));
    return JAERO_OK;
}

int64_t jaero_chan_launch_count(const jaero_chan *c) { return c ? c->launches : 0; }

int jaero_chan_write_device(jaero_chan *c, const void *d_iq, size_t n)
{
    if (!c || (!d_iq && n)) { set_error("jaero_chan_write_device: null argument"); return JAERO_E_ARG; }
    if (n > ((size_t)1 << 31)) { set_error("jaero_chan_write_device: at most 2^31 samples per write"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    const long long N0 = c->n_in, D = c->D;
    const long long m_first = (N0 + D - 1) / D, m_end = (N0 + (long long)n + D - 1) / D;
    const size_t M = (size_t)(m_end - m_first);
    c->n_out = M;
    if (n == 0) return JAERO_OK;
    const int nb = 1 - c->cur;
    const size_t need = (size_t)c->H + n;
    if (c->x[nb].reserve(need, c->stream)) return JAERO_E_CUDA;
    if (M > 0) {
        if (c->out.reserve(((M + 7) & ~(size_t)7) * c->C, c->stream)) return JAERO_E_CUDA;
        c->stride = c->out.cap / c->C;
    }
    const long long tot = c->H + (long long)n;
    chan_convert_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, c->stream>>>(d_iq, c->fmt, (long long)n,
                                                                              c->have_prev ? c->x[c->cur].ptr : nullptr, c->last_n, c->H, c->x[nb].ptr);
    JB_CUDA(cudaGetLastError());
    c->launches++;
    if (M > 0) {
        dim3 grid((unsigned)((M + TILE_M - 1) / TILE_M), (unsigned)(c->Cpad / TILE_C));
        const long long off0 = m_first * D - N0 + c->H;
        chan_ddc_kernel<<<grid, THREADS, 0, c->stream>>>(c->d_G, c->Cpad, c->Tpad, c->C, c->x[nb].ptr, off0, c->D, (int)M,
                                                         (unsigned long long)m_first, c->d_inc, c->inc_a, c->gain, c->out.ptr, c->stride);
        JB_CUDA(cudaGetLastError());
        c->launches++;
    }
    c->cur = nb; c->last_n = (long long)n; c->have_prev = true;
    c->n_in = N0 + (long long)n;
    return JAERO_OK;
}

int jaero_chan_write(jaero_chan *c, const void *iq, size_t n)
{
    if (!c || (!iq && n)) { set_error("jaero_chan_write: null argument"); return JAERO_E_ARG; }
    if (n > ((size_t)1 << 31)) { set_error("jaero_chan_write: at most 2^31 samples per write"); return JAERO_E_ARG; }
    if (n == 0) return jaero_chan_write_device(c, nullptr, 0);
    JB_CUDA(cudaSetDevice(c->device));
    const size_t bytes = n * (c->fmt == JAERO_IQ_CS16 ? 4 : 2);
    if (c->raw.reserve(bytes, c->stream)) return JAERO_E_CUDA;
    JB_CUDA(cudaMemcpyAsync(c->raw.ptr, iq, bytes, cudaMemcpyHostToDevice, c->stream));
    return jaero_chan_write_device(c, c->raw.ptr, n);
}

int jaero_chan_output_device(jaero_chan *c, const int16_t **d_pcm, size_t *n_samples, size_t *channel_stride)
{
    if (!c || !d_pcm || !n_samples || !channel_stride) { set_error("jaero_chan_output_device: null argument"); return JAERO_E_ARG; }
    *d_pcm = c->out.ptr; *n_samples = c->n_out; *channel_stride = c->stride;
    return JAERO_OK;
}

int jaero_chan_read(jaero_chan *c, int16_t *out, size_t cap, size_t *n_samples)
{
    if (!c || !out || !n_samples) { set_error("jaero_chan_read: null argument"); return JAERO_E_ARG; }
    if (cap < c->n_out) { set_error("jaero_chan_read: cap_per_channel is smaller than the output"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    *n_samples = c->n_out;
    if (c->n_out)
        JB_CUDA(cudaMemcpy2DAsync(out, cap * sizeof(int16_t), c->out.ptr, c->stride * sizeof(int16_t), c->n_out * sizeof(int16_t), c->C,
                                  cudaMemcpyDeviceToHost, c->stream));
    JB_CUDA(cudaStreamSynchronize(c->stream));
    return JAERO_OK;
}

} // extern "C"
