// C ABI of the burst demodulators (jaero_burst_*): creation from the host design (host_design.h), the per-channel helper
// kernels and the chunked write path (Hilbert transform, acquisition, trident FFTs, demodulation).
#include "capi_internal.cuh"
#include "host_design.h"
#include <algorithm>
#include <cstring>

using namespace jb;

namespace {
__global__ void burst_init_kernel(BurstParams p, double freq_center, double st_freq)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.cpad) return;
    auto D = [&](int i) -> double & { return p.BD[(size_t)i * p.cpad + ch]; };
    auto I = [&](int i) -> int & { return p.BI[(size_t)i * p.cpad + ch]; };
    const double sr = (double)((float)((int)p.Fs));
    D(BD_M2_FREQ) = freq_center; D(BD_M2_STEP) = (freq_center) * ((double)jb::WTSIZE) / sr;
    D(BD_MC_FREQ) = freq_center; D(BD_MC_STEP) = (freq_center) * ((double)jb::WTSIZE) / sr;
    D(BD_ST_FREQ) = st_freq; D(BD_ST_STEP) = (st_freq) * ((double)jb::WTSIZE) / sr;
    D(BD_SH_FREQ) = st_freq; D(BD_SH_STEP) = (st_freq) * ((double)jb::WTSIZE) / sr;
    D(BD_MSE) = 10.0;                                    // burstmskdemodulator.cpp:195
    D(BD_ROT_RE) = 1.0; D(BD_SAV_RE) = 1.0;              // rotator=1, symboltone_averotator=1 (:201-202); symboltone_rotator stays 0
    D(BD_DIFF_LAST) = -1.0;
    if (p.kind == 1) {                                   // burst OQPSK ctor (burstoqpskdemodulator.cpp:4-133)
        D(BD_MSE) = 100.0; D(BD_VOL_GAIN) = 1.0; D(BD_STR_RE) = 1.0;     // symboltone_rotator=1, never reset
        D(BD_ST_FREQ) = 10500.0; D(BD_ST_STEP) = (10500.0) * ((double)jb::WTSIZE) / sr;
        D(BD_SR_FREQ) = 10500.0; D(BD_SR_STEP) = (10500.0) * ((double)jb::WTSIZE) / sr;
        D(BD_SH_FREQ) = 10500.0 / 4.0; D(BD_SH_STEP) = (10500.0 / 4.0) * ((double)jb::WTSIZE) / sr;
    }
    I(BI_PD_CNTDOWN) = 2 * p.pd_len; I(BI_PD_MAXPOSCNT) = -1;    // PeakDetector::setSettings (DSP.h:502-513)
    I(BI_STARTSTOP) = -1;                                // ctor :69
}
__global__ void burst_soft_reset_kernel(BurstParams p)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels) return;
    int &count = p.BI[(size_t)BI_SOFT_COUNT * p.cpad + ch];
    const int pending = p.BI[(size_t)BI_SOFT_PENDING * p.cpad + ch];
    int16_t *ring = p.soft + (size_t)ch * p.soft_cap;
    for (int k = 0; k < pending; k++) ring[k] = ring[count + k];
    count = 0;
}
__global__ void burst_set_int_kernel(BurstParams p, int idx, int channel, int value)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels) return;
    if (channel < 0 || channel == ch) p.BI[(size_t)idx * p.cpad + ch] = value;
}
} // namespace

int jb::burst_soft_reset(const jaero_burst *b, cudaStream_t s)
{
    burst_soft_reset_kernel<<<(b->p.n_channels + 127) / 128, 128, 0, s>>>(b->p);
    JB_CUDA(cudaGetLastError());
    return JAERO_OK;
}

static int burst_create(const jaero_settings *s, int n_channels, int device, int kind, jaero_burst **out)
{
    BurstPlan plan;
    const char *bad = out ? burst_plan(s, n_channels, kind, plan) : "jaero_burst_create: bad argument";
    if (bad) { set_error(bad); return JAERO_E_ARG; }
    NewHandle<jaero_burst> nh(jaero_burst_destroy);
    int r = nh.open(device, "jaero_burst_msk_create"); if (r) return r;
    jaero_burst *b = nh.h;
    HandleAllocs &A = b->allocs;
    cudaStream_t st = b->stream;
    BurstParams &p = b->p;
    p = plan.p;
    const size_t cp = p.cpad, C = n_channels;
    int rc = 0;
    rc |= A.zeroed(&p.BD, (size_t)BD_COUNT * cp, st); rc |= A.zeroed(&p.BI, (size_t)BI_COUNT * cp, st);
    rc |= A.zeroed(&p.agc_ring, (size_t)p.agc_len * cp, st); rc |= A.zeroed(&p.d1_ring, (size_t)p.d1_len * cp, st);
    rc |= A.zeroed(&p.d2_ring, (size_t)p.d2_len * cp, st); rc |= A.zeroed(&p.btd1_ring, (size_t)p.btd1_len * cp, st);
    rc |= A.zeroed(&p.btma_ring, (size_t)p.btma_len * cp, st); rc |= A.zeroed(&p.mav1_ring, (size_t)p.mav1_len * cp, st);
    rc |= A.zeroed(&p.btdiff_ring, (size_t)p.btdiff_len * cp, st);
    rc |= A.zeroed(&p.pd1_ring, (size_t)(2 * p.pd_len + 1) * cp, st); rc |= A.zeroed(&p.pd2_ring, (size_t)(p.pd_len + 1) * cp, st);
    rc |= A.zeroed(&p.pd3_ring, (size_t)(2 * p.pd_len + 1) * cp, st);
    rc |= A.zeroed(&p.a1_ring, (size_t)(p.a1_k + 1) * cp, st); rc |= A.zeroed(&p.eb1_ring, (size_t)p.eb_len * cp, st);
    rc |= A.zeroed(&p.eb2_ring, (size_t)p.eb_len * cp, st); rc |= A.zeroed(&p.agc2_ring, (size_t)p.agc2_len * cp, st);
    rc |= A.zeroed(&p.d8_ring, (size_t)(p.d8_k + 1) * cp, st); rc |= A.zeroed(&p.msema_ring, (size_t)p.msema_len * cp, st);
    rc |= A.zeroed(&p.fir_re, (size_t)(p.ntaps + 1) * cp, st); rc |= A.zeroed(&p.fir_im, (size_t)(p.ntaps + 1) * cp, st);
    rc |= A.zeroed(&p.ds_ring, (size_t)p.ds_len * cp, st);
    rc |= A.zeroed(&p.tri, C * BURST_MAXEV * p.tri_sz, st); rc |= A.zeroed(&p.ev_sample, C * BURST_MAXEV, st);
    rc |= A.zeroed(&p.ev_result, C * BURST_MAXEV * 8, st);
    rc |= A.zeroed(&p.analytic, C * p.astride, st); rc |= A.zeroed(&p.vtd, C * p.astride, st);
    rc |= A.zeroed(&p.soft, C * p.soft_cap, st);
    {
        double *d1 = 0, *d2 = 0, *d3 = 0;
        rc |= A.upload(&d1, plan.w_btd1, st); rc |= A.upload(&d2, plan.w_btdiff, st); rc |= A.upload(&d3, plan.w_a1, st);
        p.btd1_wv = d1; p.btdiff_wv = d2; p.a1_wv = d3;
    }
    HilbertStream &h = b->hil;
    h = plan.hil;
    rc |= A.upload(&h.H, plan.hil_H, st); rc |= A.upload(&h.tw, plan.hil_tw, st);
    rc |= A.zeroed(&h.hist, C * (h.K - 1), st); rc |= A.zeroed(&h.inblk, C * h.L, st); rc |= A.zeroed(&h.outblk, C * h.L, st);
    b->ev_round = 128;
    rc |= A.upload(&b->tw32k, plan.tw32k, st);
    rc |= A.zeroed(&b->wa, (size_t)2 * b->ev_round * TRI_N, st); rc |= A.zeroed(&b->wb, (size_t)2 * b->ev_round * TRI_N, st);
    rc |= A.zeroed(&b->d_ev_list, (size_t)2 * C * BURST_MAXEV, st);
    {
        std::vector<double> sn, cs;
        trig_tables(sn, cs);
        double *ds = 0, *dc = 0;
        rc |= A.upload(&ds, sn, st); rc |= A.upload(&dc, cs, st);
        p.sin_t = ds; p.cos_t = dc;
    }
    if (rc) return JAERO_E_CUDA;
    burst_init_kernel<<<(p.cpad + 127) / 128, 128, 0, st>>>(p, plan.freq_center, p.fb / 2.0);
    JB_CUDA(cudaGetLastError());
    if (A.pinned(&b->h_ints, (size_t)BI_COUNT * cp) || A.pinned(&b->h_dbls, (size_t)BD_COUNT * cp) || A.pinned(&b->h_soft, C * p.soft_cap))
        return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(st));
    *out = nh.release();
    return JAERO_OK;
}

extern "C" {

int jaero_burst_msk_create(const jaero_settings *s, int n_channels, int device, jaero_burst **out) { return burst_create(s, n_channels, device, 0, out); }
int jaero_burst_oqpsk_create(const jaero_settings *s, int n_channels, int device, jaero_burst **out) { return burst_create(s, n_channels, device, 1, out); }
void jaero_burst_destroy(jaero_burst *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    cudaStreamSynchronize(b->stream);
    b->allocs.free_all(); b->stage.release();
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
}
int64_t jaero_burst_launch_count(const jaero_burst *b) { return b ? b->launches : 0; }
int jaero_burst_sync(jaero_burst *b)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    return JAERO_OK;
}
int jaero_burst_write_device(jaero_burst *b, const int16_t *d_pcm, size_t n, size_t stride)
{
    if (!b || !d_pcm) { set_error("jaero_burst_write_device: null argument"); return JAERO_E_ARG; }
    if (n == 0) return JAERO_OK;
    if (stride < n || n > 0x7fffffff) { set_error("jaero_burst_write_device: bad stride / length"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const BurstParams &p = b->p;
    const size_t cp = p.cpad;
    int new_write = 1;
    for (size_t c0 = 0; c0 < n; c0 += BURST_CHUNK) {
        const int m = (int)std::min((size_t)BURST_CHUNK, n - c0);
        // Hilbert transform of this chunk (JFastFir::update: per-sample exchange + block transforms)
        int i = 0;
        while (i < m) {
            const int take = std::min(b->hil.L - b->hil_fill, m - i);
            if (hilbert_exchange_launch(b->hil, p, d_pcm, stride, (int)c0, i, i + take, b->hil_fill, b->stream)) return JAERO_E_CUDA;
            b->launches++;
            b->hil_fill += take; i += take;
            if (b->hil_fill == b->hil.L) {
                if (hilbert_block_launch(b->hil, p.n_channels, b->hil_blocks == 0 ? 1 : 0, b->stream)) return JAERO_E_CUDA;
                b->launches++; b->hil_fill = 0; b->hil_blocks++;
            }
        }
        if (burst_front_launch(p, b->samples, m, b->stream)) return JAERO_E_CUDA;
        b->launches++;
        // trident events of this chunk
        JB_CUDA(cudaMemcpyAsync(b->h_ints, p.BI + (size_t)BI_NEV * cp, cp * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
        JB_CUDA(cudaStreamSynchronize(b->stream));
        b->h_ev.clear();
        for (int ch = 0; ch < p.n_channels; ch++) for (int e = 0; e < b->h_ints[ch]; e++) { b->h_ev.push_back(ch); b->h_ev.push_back(e); }
        const int nevt = (int)b->h_ev.size() / 2;
        if (nevt) JB_CUDA(cudaMemcpyAsync(b->d_ev_list, b->h_ev.data(), b->h_ev.size() * sizeof(int), cudaMemcpyHostToDevice, b->stream));
        for (int e0 = 0; e0 < nevt; e0 += b->ev_round) {
            const int cnt = std::min(b->ev_round, nevt - e0);
            if (burst_trident_fft_launch(p, b->d_ev_list + 2 * e0, cnt, b->wa, b->wb, b->tw32k, b->stream)) return JAERO_E_CUDA;
            b->launches += 2;
        }
        if (burst_back_launch(p, b->samples, m, new_write, b->stream)) return JAERO_E_CUDA;
        new_write = 0;
        b->launches++;
        b->samples += m;
    }
    return JAERO_OK;
}
int jaero_burst_write(jaero_burst *b, const int16_t *pcm, size_t n, size_t stride)
{
    if (!b || !pcm) { set_error("jaero_burst_write: null argument"); return JAERO_E_ARG; }
    if (n == 0) return JAERO_OK;
    if (stride < n) { set_error("jaero_burst_write: channel_stride < n_samples"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const size_t C = b->p.n_channels, pitch = (n + 7) & ~(size_t)7;
    if (b->stage.reserve(C * pitch, b->stream)) return JAERO_E_CUDA;
    JB_CUDA(cudaMemcpy2DAsync(b->stage.ptr, pitch * 2, pcm, stride * 2, n * 2, C, cudaMemcpyHostToDevice, b->stream));
    return jaero_burst_write_device(b, b->stage.ptr, n, pitch);
}
int jaero_burst_read_softbits(jaero_burst *b, int16_t *out, size_t cap, int32_t *counts)
{
    if (!b || !out || !counts) { set_error("jaero_burst_read_softbits: null argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const BurstParams &p = b->p; const size_t cp = p.cpad;
    JB_CUDA(cudaMemcpyAsync(b->h_ints, p.BI, (size_t)BI_COUNT * cp * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    const int *cnt = b->h_ints + (size_t)BI_SOFT_COUNT * cp, *ovf = b->h_ints + (size_t)BI_SOFT_OVERFLOW * cp;
    const int r = read_soft_rows(cnt, ovf, p.n_channels, p.soft, p.soft_cap, b->h_soft, out, cap, counts, b->stream);
    return r ? r : burst_soft_reset(b, b->stream);
}
int jaero_burst_set_dcd(jaero_burst *b, int channel, int dcd)
{
    if (!b || channel >= b->p.n_channels) { set_error("jaero_burst_set_dcd: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    burst_set_int_kernel<<<(b->p.n_channels + 127) / 128, 128, 0, b->stream>>>(b->p, BI_DCD, channel, dcd ? 1 : 0);
    JB_CUDA(cudaGetLastError());
    return JAERO_OK;
}
int jaero_burst_set_afc(jaero_burst *b, int state)                  // burstmskdemodulator.cpp / burstoqpskdemodulator.cpp setAFC
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    b->p.afc = state ? 1 : 0;
    return JAERO_OK;
}
int jaero_burst_set_sql(jaero_burst *b, int state)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    b->p.sql = state ? 1 : 0;
    return JAERO_OK;
}
int jaero_burst_get_status_all(jaero_burst *b, jaero_burst_status *out)
{
    if (!b || !out) { set_error("null argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const size_t cp = b->p.cpad;
    JB_CUDA(cudaMemcpyAsync(b->h_dbls, b->p.BD, (size_t)BD_COUNT * cp * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
    JB_CUDA(cudaMemcpyAsync(b->h_ints, b->p.BI, (size_t)BI_COUNT * cp * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    for (int ch = 0; ch < b->p.n_channels; ch++) {
        auto D = [&](int i) { return b->h_dbls[(size_t)i * cp + ch]; };
        auto I = [&](int i) { return b->h_ints[(size_t)i * cp + ch]; };
        jaero_burst_status &s = out[ch];
        s.mixer2_freq = D(BD_M2_FREQ); s.mixer2_wtptr = D(BD_M2_PTR); s.center_freq = D(BD_MC_FREQ); s.st_freq = D(BD_ST_FREQ); s.st_wtptr = D(BD_ST_PTR);
        s.agc = D(BD_AGC_VAL); s.mse = D(BD_MSE); s.ebno = D(BD_EB_EBNO); s.vol_gain = D(BD_VOL_GAIN); s.rotator_freq = D(BD_ROT_FREQ);
        s.n_sig_true = I(BI_SIG_TRUE); s.n_sig_false = I(BI_SIG_FALSE); s.cntr = I(BI_CNTR); s.startstop = I(BI_STARTSTOP);
        s.last_burst_ebno = D(BD_LAST_EBNO_EMIT); s.n_ebno_emits = I(BI_EBNO_EMITS);
    }
    return JAERO_OK;
}
} // extern "C"
