// Device channelizer (include/jaero_b200.h, "device channelizer"): one wideband complex IQ stream in, one real int16 audio
// row per channel out, in the layout jaero_batch_write_device consumes.
//
// The rate change is L/M (L = 1 for an integer ratio D = M). Output m sits at input time mM/L: n_m = floor(mM/L), polyphase
// branch p_m = mM mod L, taps h[kL + p_m]. phi_c(n - k) = phi_c(n) - phi_c(k) holds exactly in uint32 phase arithmetic, so the
// mix-to-0-Hz, low-pass and resample of every channel is one complex matrix product per branch, shared by all channels:
//   A[c][m] = sum_k G[p_m][k][c] X[k][m],   G[p][k][c] = h[kL + p] e^{+2 pi j phi_c(k) / 2^32},   X[k][m] = x[n_m - k],
// followed per output by one rotation through (psi(m) - phi_c(n_m)) mod 2^32, the gain, rounding and saturation.
// The outputs m = m_r + jL of one residue class share the branch and step through the input by exactly M, so each class is
// an integer-stride decimation; one launch covers all classes (blockIdx.z). G is built once at create (double, stored as
// float2); x is kept as float2 behind a copy of the last Tpad-1 input samples (shared by all channels; channels carry no
// other state). chan_ddc_kernel runs k in a fixed ascending order for every output, so each output's sum does not depend
// on how the input was cut into writes.
#include "../../include/jaero_b200.h"
#include "handle.cuh"
#include <cmath>
#include <algorithm>
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

// One block: TILE_C channels x TILE_M outputs of residue class q = blockIdx.z, i.e. outputs m = m_first + q + jL. G is
// [L][Tpad][Cpad] (branch-major, then tap-major, zero beyond Tp and C). The class starts at m_r = m_first + q, input index
// n_r = floor(m_r Dm / L), branch p = m_r Dm mod L; its local output j reads xb[pos], pos = n_r + hist + j*Dm - k
// (hist = H - N0: where input index n lies in xb), and goes to out[c*stride + q + j*L]. With L = 1 this is the integer-D
// decimation: one class, p = 0, n_r = m_first * D.
__global__ void __launch_bounds__(THREADS) chan_ddc_kernel(const float2 *__restrict__ G, int Cpad, int Tpad, int C,
                                                           const float2 *__restrict__ xb, long long hist, int Dm, int L,
                                                           int n_out, unsigned long long m_first, const uint32_t *__restrict__ inc_c,
                                                           uint32_t inc_a, double gain, int16_t *__restrict__ out, size_t stride)
{
    __shared__ float2 Gs[KC][TILE_C];
    __shared__ float2 Xs[KC][TILE_M + 1];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int q = blockIdx.z, c0 = blockIdx.y * TILE_C, j0 = blockIdx.x * TILE_M;
    const int M = (n_out - q + L - 1) / L;                                   // outputs of this class in this write
    if (j0 >= M) return;
    const unsigned long long m_r = m_first + q, t_r = m_r * (unsigned long long)Dm;
    const unsigned long long n_r = t_r / (unsigned)L;
    const int p = (int)(t_r % (unsigned)L);
    const long long off0 = (long long)n_r + hist;
    G += (size_t)p * Tpad * Cpad;
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
            Xs[kk][mm] = j < M ? xb[off0 + (long long)j * Dm - (k0 + kk)] : make_float2(0.f, 0.f);
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
            uint32_t phi = ic * (uint32_t)(n_r + (unsigned long long)jj * Dm);   // phi_c(n_m), mod 2^32
            uint32_t psi = inc_a * (uint32_t)(m_r + (unsigned long long)jj * L);
            int32_t th = (int32_t)(psi - phi);
            double s, co;
            sincospi((double)th * (1.0 / 2147483648.0), &s, &co);
            double v = gain * ((double)acc[i][j].x * co - (double)acc[i][j].y * s);
            v = rint(v);
            v = fmin(fmax(v, -32768.0), 32767.0);
            out[(size_t)c * stride + q + (size_t)jj * L] = (int16_t)v;
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

// Validates the settings, finds L/M = output_rate / input_rate in lowest terms (the smallest L in 1..64 for which r L,
// r = input_rate / output_rate, is within 1e-9 r L of an integer M; M >= 2L) and designs the prototype h at L * input_rate:
// scipy.signal.firwin(T, (f_p + f_s)/2, window=('kaiser', beta), fs=L*input_rate) * L with T from
// kaiserord(60, (f_s - f_p) / (L*input_rate / 2)), made odd, and at most 8191 taps per branch (ceil(T/L)). Returns T or
// JAERO_E_ARG.
int chan_design(const jaero_chan_settings *s, std::vector<double> *h, int *L_out, int *M_out)
{
    if (!s) { set_error("jaero_chan: null settings"); return JAERO_E_ARG; }
    if (s->iq_format != JAERO_IQ_CS16 && s->iq_format != JAERO_IQ_CU8) { set_error("jaero_chan: unknown iq_format"); return JAERO_E_ARG; }
    if (!std::isfinite(s->input_rate) || !std::isfinite(s->output_rate) || s->input_rate <= 0 || s->output_rate <= 0) {
        set_error("jaero_chan: input_rate and output_rate must be positive"); return JAERO_E_ARG; }
    double r = s->input_rate / s->output_rate;
    int L = 0;
    double Md = 0;
    for (int l = 1; l <= JAERO_CHAN_MAX_PHASES && !L; l++) {
        double rl = r * l, m = std::floor(rl + 0.5);
        if (std::fabs(rl - m) <= 1e-9 * rl) { L = l; Md = m; }
    }
    if (!L || Md < 2 * L || Md > 1e6 * L) {
        set_error("jaero_chan: output_rate / input_rate must be L/M with L <= 64 and M >= 2L"); return JAERO_E_ARG; }
    if (!std::isfinite(s->audio_hz) || s->audio_hz <= 0 || s->audio_hz >= 0.5 * s->output_rate) {
        set_error("jaero_chan: audio_hz must lie in (0, output_rate/2)"); return JAERO_E_ARG; }
    if (!std::isfinite(s->passband_hz) || s->passband_hz <= 0) { set_error("jaero_chan: passband_hz must be positive"); return JAERO_E_ARG; }
    if (!std::isfinite(s->gain) || s->gain <= 0) { set_error("jaero_chan: gain must be positive and finite"); return JAERO_E_ARG; }
    const double A = 60.0, fsamp = L * s->input_rate;
    double fp = 0.5 * s->passband_hz;
    double fs = std::fmin(2 * s->audio_hz, s->output_rate - 2 * s->audio_hz) - fp;
    if (!(fs > fp)) { set_error("jaero_chan: no transition band (f_s <= f_p): narrow the passband or move audio_hz"); return JAERO_E_ARG; }
    double width = (fs - fp) / (0.5 * fsamp);
    double numtaps = (A - 7.95) / 2.285 / (M_PI * width) + 1;
    if (!(numtaps <= (double)JAERO_CHAN_MAX_TAPS * L)) { set_error("jaero_chan: filter longer than 8191 taps per phase"); return JAERO_E_ARG; }
    int T = (int)std::ceil(numtaps);
    if (!(T & 1)) T++;
    if ((T + L - 1) / L > JAERO_CHAN_MAX_TAPS) { set_error("jaero_chan: filter longer than 8191 taps per phase"); return JAERO_E_ARG; }
    if (h) {
        const double beta = 0.1102 * (A - 8.7), cut = (fp + fs) / 2 / (0.5 * fsamp), alpha = 0.5 * (T - 1);
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
        for (int n = 0; n < T; n++) (*h)[n] = (*h)[n] / sum * L;   // sum L: unity DC gain in every branch
    }
    if (L_out) *L_out = L;
    if (M_out) *M_out = (int)Md;
    return T;
}

} // namespace

struct jaero_chan {
    int device, C, Cpad, T, Tpad, H, L, M, fmt;                      // Tpad: taps per branch, ceil(T/L) rounded up to KC
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
    int T = chan_design(s, taps ? &h : nullptr, nullptr, nullptr);
    if (T < 0) return T;
    if (taps)
        for (int k = 0; k < T && k < cap; k++) taps[k] = h[k];
    return T;
}

int jaero_chan_ratio(const jaero_chan_settings *s, int *L, int *M)
{
    int l = 0, m = 0;
    int T = chan_design(s, nullptr, &l, &m);
    if (T < 0) return T;
    if (L) *L = l;
    if (M) *M = m;
    return JAERO_OK;
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
    int L = 0, M = 0;
    int T = chan_design(s, &h, &L, &M);
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
    c->C = n_channels; c->T = T; c->L = L; c->M = M; c->fmt = s->iq_format; c->gain = s->gain;
    const int Tp = (T + L - 1) / L;
    c->Cpad = (n_channels + TILE_C - 1) / TILE_C * TILE_C;
    c->Tpad = (Tp + KC - 1) / KC * KC;
    c->H = c->Tpad - 1;
    c->inc_a = (uint32_t)(int64_t)llround(s->audio_hz / s->output_rate * 4294967296.0);
    std::vector<uint32_t> inc(n_channels);
    for (int k = 0; k < n_channels; k++) inc[k] = (uint32_t)(int64_t)llround(offset_hz[k] / s->input_rate * 4294967296.0);
    const size_t branch = (size_t)c->Tpad * c->Cpad;
    std::vector<float2> G(branch * L, make_float2(0.f, 0.f));
    for (int k = 0; k < Tp; k++)
        for (int ch = 0; ch < n_channels; ch++) {
            uint32_t ph = inc[ch] * (uint32_t)k;
            double a = 2.0 * M_PI * (double)ph / 4294967296.0, co = std::cos(a), si = std::sin(a);
            for (int p = 0; p < L && k * L + p < T; p++) {
                double hk = h[k * L + p];
                G[p * branch + (size_t)k * c->Cpad + ch] = make_float2((float)(hk * co), (float)(hk * si));
            }
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
    const long long N0 = c->n_in, L = c->L, Md = c->M;
    const long long m_first = (L * N0 + Md - 1) / Md, m_end = (L * (N0 + (long long)n) + Md - 1) / Md;   // n_m inside the input
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
        const size_t per_class = (M + L - 1) / L;                   // outputs of residue class 0, the largest
        dim3 grid((unsigned)((per_class + TILE_M - 1) / TILE_M), (unsigned)(c->Cpad / TILE_C), (unsigned)std::min<size_t>(L, M));
        chan_ddc_kernel<<<grid, THREADS, 0, c->stream>>>(c->d_G, c->Cpad, c->Tpad, c->C, c->x[nb].ptr, c->H - N0, c->M, c->L, (int)M,
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
