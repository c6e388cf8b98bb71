// C ABI of the continuous demodulator batches (jaero_batch_*): creation from the host design (host_design.h), the
// per-channel helper kernels, the seating of the pipelined 10500 bps kernel and the write path that cuts a call into
// segment launches at the coarse-estimator triggers.
#include "capi_internal.cuh"
#include "host_design.h"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

using namespace jb;

namespace {

__global__ void init_state_kernel(DemodParams p, const double *freq_center, double st_freq, double ebno_init)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels) return;
    auto D = [&](int i) -> double & { return p.D[(size_t)i * p.cpad + ch]; };
    auto I = [&](int i) -> int & { return p.I[(size_t)i * p.cpad + ch]; };
    // WaveTable::SetFreq(double,int) (DSP.cpp:142-149): WTstep = freq*WTSIZE/(float)samplerate
    double fc = freq_center[ch];
    if (fc > ((p.Fs / 2.0) - (p.lockingbw / 2.0))) fc = ((p.Fs / 2.0) - (p.lockingbw / 2.0));   // oqpskdemodulator.cpp:183
    if (fc < 0) fc = 0;
    const double sr = (double)((float)((int)p.Fs));
    D(D_M2_FREQ) = fc; D(D_M2_STEP) = (fc) * ((double)jb::WTSIZE) / sr;
    D(D_MC_FREQ) = fc; D(D_MC_STEP) = (fc) * ((double)jb::WTSIZE) / sr;
    D(D_ST_FREQ) = st_freq; D(D_ST_STEP) = (st_freq) * ((double)jb::WTSIZE) / sr;
    D(D_SR_FREQ) = st_freq; D(D_SR_STEP) = (st_freq) * ((double)jb::WTSIZE) / sr;
    D(D_MSE) = (p.kind == JAERO_KIND_OQPSK) ? 100.0 : 10.0;       // oqpskdemodulator.cpp:17 / mskdemodulator.cpp:180
    D(D_DIFF_LAST) = -1.0;                                        // DSP.cpp:520
    D(D_EB_EBNO) = ebno_init;
    I(I_COUNTDOWN) = 4; I(I_COUNTDOWN2) = 5;                      // oqpskdemodulator.cpp:641,652 / mskdemodulator.cpp:493
    I(I_EMPTYING) = 1;                                            // coarsefreqestimate.cpp:24
}

// after a host read: move the not-yet-emitted (<32 / <12) soft bits to the front of each ring
__global__ void soft_reset_kernel(DemodParams p)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels) return;
    int &count = p.I[(size_t)I_SOFT_COUNT * p.cpad + ch];
    const int pending = p.I[(size_t)I_SOFT_PENDING * p.cpad + ch];
    int16_t *ring = p.soft + (size_t)ch * p.soft_cap;
    for (int k = 0; k < pending; k++) ring[k] = ring[count + k];
    p.soft_total[ch] += count;
    count = 0;
    p.I[(size_t)I_LOST_N * p.cpad + ch] = 0;             // the frame layer consumed the events before the ring is reset
}
__global__ void set_int_kernel(DemodParams p, int idx, int channel, int value)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels) return;
    if (channel < 0 || channel == ch) p.I[(size_t)idx * p.cpad + ch] = value;
}
// PeakVolume (oqpskdemodulator.cpp:393-405, mskdemodulator.cpp:329-344): max |sample| of the input since the last read-out.
// One warp per channel row, 16-byte loads; the same for every demodulator kernel variant.
__global__ void peak_kernel(DemodParams p, const int16_t *__restrict__ pcm, size_t stride, int n)
{
    const int ch = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (ch >= p.n_channels) return;
    const int4 *row = reinterpret_cast<const int4 *>(pcm + (size_t)ch * stride);
    int m = 0;
    for (int k = lane; k * 8 < n; k += 32) {
        const int4 v = __ldg(row + k);
        const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int lo = (int)(short)(w[q] & 0xffff), hi = w[q] >> 16;
            if (k * 8 + 2 * q < n) m = max(m, abs(lo));
            if (k * 8 + 2 * q + 1 < n) m = max(m, abs(hi));
        }
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if (lane == 0) { int &pk = p.I[(size_t)I_PEAK * p.cpad + ch]; pk = max(pk, m); }
}
// CenterFreqChangedSlot (oqpskdemodulator.cpp:291-310 / mskdemodulator.cpp:265-282)
__global__ void center_freq_kernel(DemodParams p, int channel, double freq_center)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels || (channel >= 0 && channel != ch)) return;
    auto D = [&](int i) -> double & { return p.D[(size_t)i * p.cpad + ch]; };
    double fc = freq_center;
    if (p.kind == JAERO_KIND_OQPSK) {
        if (p.fb != 8400) { if (fc < (0.5 * p.fb)) fc = 0.5 * p.fb; if (fc > (p.Fs / 2.0 - 0.5 * p.fb)) fc = p.Fs / 2.0 - 0.5 * p.fb; }
    } else { if (fc < (0.75 * p.fb)) fc = 0.75 * p.fb; if (fc > (p.Fs / 2.0 - 0.75 * p.fb)) fc = p.Fs / 2.0 - 0.75 * p.fb; }
    if (fc < 0) fc = 0;
    const double srf = (double)((float)((int)p.Fs));
    D(D_MC_FREQ) = fc; D(D_MC_STEP) = (fc) * ((double)jb::WTSIZE) / srf;   // SetFreq(freq,Fs)
    auto set_m2 = [&](double f) { if (f < 0) f = 0; D(D_M2_FREQ) = f; D(D_M2_STEP) = (f) * ((double)jb::WTSIZE) / p.Fs; };
    if (p.afc) set_m2(D(D_MC_FREQ));
    if ((D(D_M2_FREQ) - D(D_MC_FREQ)) > (p.lockingbw / 2.0)) set_m2(D(D_MC_FREQ) + (p.lockingbw / 2.0));
    if ((D(D_M2_FREQ) - D(D_MC_FREQ)) < (-p.lockingbw / 2.0)) set_m2(D(D_MC_FREQ) - (p.lockingbw / 2.0));
    double2 *row = p.bb + (size_t)ch * p.bb_len;
    for (int j = 0; j < p.bb_len; j++) row[j] = make_double2(0.0, 0.0);
}
// ---- seating by symbol-timing phase (pipelined 10500 bps kernel)
// key[c] = samples until channel c's next carrier-update strobe, in [0, 2 * samples per strobe): st_osc passes the point ee
// (oqpskdemodulator.cpp:488) every Fs/fb samples and every second passage (yui, :496-503) is a carrier update.
__global__ void regroup_key_kernel(DemodParams p, double *__restrict__ key)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_channels) return;
    const double ptr = p.D[(size_t)D_ST_PTR * p.cpad + ch], step = p.D[(size_t)D_ST_STEP * p.cpad + ch];
    const int yui = p.I[(size_t)I_YUI * p.cpad + ch];
    const double N = (double)jb::WTSIZE;
    double d = p.ee * N - ptr; if (d < 0) d += N;
    const double per = step > 0 ? N / step : 1.0;
    double k = step > 0 ? d / step : 0.0;
    if (yui) k += per;                                    // the next passage only stores pt_d; the one after it updates the carrier
    key[ch] = fmod(k, 2.0 * per);
}
// ring_new[(cta', k, lane')] = ring_old[(cta, k, lane)] for the channel that moves from seat (cta, lane) to (cta', lane')
__global__ void regroup_ring_kernel(const double *__restrict__ src, double *__restrict__ dst, const int *__restrict__ old_seat_of_new, int len, int n_ctas)
{
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);      // (cta', k)
    if (row >= (long long)n_ctas * len) return;
    const int cta_n = (int)(row / len), k = (int)(row % len);
    const int so = old_seat_of_new[cta_n * 32 + lane];
    dst[row * 32 + lane] = src[((size_t)(so >> 5) * len + k) * 32 + (so & 31)];
}

// New seating: slot_of[c] for every channel (pads keep their seats). The rings follow; everything else is indexed by channel.
int batch_apply_seating(jaero_batch *b, const std::vector<int> &new_slot_of)
{
    DemodParams &p = b->p;
    const int cp = p.cpad, n_ctas = cp / 32;
    std::vector<int> old_seat_of_new(cp), chan_of(cp);
    for (int c = 0; c < cp; c++) { old_seat_of_new[new_slot_of[c]] = b->slot_of[c]; chan_of[new_slot_of[c]] = c; }
    const size_t need = (size_t)p.agc_len * cp;
    if (!b->d_ring_scratch) {
        if (cudaMalloc(&b->d_ring_scratch, need * sizeof(double)) != cudaSuccess) { cudaGetLastError(); b->d_ring_scratch = 0; b->regroup_every = 0; return 0; }   // no room: keep the seating
        b->allocs.dev.push_back(b->d_ring_scratch);
    }
    int *d_map = b->d_chan_of + cp;                          // second half of the allocation: old seat of each new seat
    JB_CUDA(cudaMemcpyAsync(d_map, old_seat_of_new.data(), cp * sizeof(int), cudaMemcpyHostToDevice, b->stream));
    auto move = [&](double *ring, int len) -> int {
        if (!ring) return 0;
        const long long rows = (long long)n_ctas * len;
        regroup_ring_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, b->stream>>>(ring, b->d_ring_scratch, d_map, len, n_ctas);
        JB_CUDA(cudaGetLastError());
        JB_CUDA(cudaMemcpyAsync(ring, b->d_ring_scratch, (size_t)rows * 32 * sizeof(double), cudaMemcpyDeviceToDevice, b->stream));
        b->launches++;
        return 0;
    };
    if (move(p.agc_ring, p.agc_len) || move(p.ebno_e1, p.ebno_len) || move(p.ebno_e2, p.ebno_len)) return -1;
    JB_CUDA(cudaMemcpyAsync(b->d_chan_of, chan_of.data(), cp * sizeof(int), cudaMemcpyHostToDevice, b->stream));
    JB_CUDA(cudaStreamSynchronize(b->stream));               // the host vectors above go out of scope
    b->slot_of = new_slot_of;
    b->regroups++;
    return 0;
}
int batch_regroup_by_phase(jaero_batch *b, bool force)
{
    DemodParams &p = b->p;
    const int C = p.n_channels, cp = p.cpad;
    regroup_key_kernel<<<(C + 127) / 128, 128, 0, b->stream>>>(p, b->d_keys);
    JB_CUDA(cudaGetLastError());
    JB_CUDA(cudaMemcpyAsync(b->h_keys, b->d_keys, C * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    b->launches++;
    // Is the present seating still coherent? A CTA is coherent when the carrier-update strobes of its channels fall within 1.5
    // samples of each other (circularly, period = two strobe intervals). Moving the rings costs ~30 ms per 4096 channels, so the
    // seating is only changed when more than a quarter of the CTAs have drifted apart (never, for transmitters on one clock).
    if (!force) {
        const double period = 2.0 * p.Fs / p.fb;                                     // keys are in [0, 2*Fs/fb)
        static const double thr = getenv("JAERO_REGROUP_SPREAD") ? atof(getenv("JAERO_REGROUP_SPREAD")) : 1.5;
        int bad = 0, ctas = 0;
        std::vector<double> ks, spreads;
        std::vector<std::vector<int>> members(cp / 32);
        for (int c = 0; c < C; c++) members[b->slot_of[c] >> 5].push_back(c);
        for (auto &m : members) {
            if (m.size() < 2) continue;
            ctas++;
            ks.clear();
            for (int c : m) ks.push_back(b->h_keys[c]);
            std::sort(ks.begin(), ks.end());
            double gap = ks.front() + period - ks.back();
            for (size_t i = 1; i < ks.size(); i++) gap = std::max(gap, ks[i] - ks[i - 1]);
            spreads.push_back(period - gap);
            if (period - gap > thr) bad++;
        }
        if (getenv("JAERO_DEBUG") && !spreads.empty()) {
            std::sort(spreads.begin(), spreads.end());
            fprintf(stderr, "[jaero_b200] seating check at epoch %lld: %d of %d CTAs spread > %.1f samples (median %.2f, p90 %.2f, max %.2f)\n", b->epochs, bad, ctas, thr,
                    spreads[spreads.size() / 2], spreads[spreads.size() * 9 / 10], spreads.back());
        }
        if (bad * 4 <= ctas) return 0;
    }
    std::vector<int> order(C);
    for (int c = 0; c < C; c++) order[c] = c;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return b->h_keys[x] < b->h_keys[y]; });
    std::vector<int> slot_of(cp);
    for (int k = 0; k < C; k++) slot_of[order[k]] = k;
    for (int c = C; c < cp; c++) slot_of[c] = c;
    if (slot_of == b->slot_of) return 0;
    return batch_apply_seating(b, slot_of);
}

} // namespace

int jb::batch_soft_reset(const jaero_batch *b, cudaStream_t s)
{
    soft_reset_kernel<<<(b->p.n_channels + 127) / 128, 128, 0, s>>>(b->p);
    JB_CUDA(cudaGetLastError());
    return JAERO_OK;
}

extern "C" {

int jaero_batch_create(const jaero_settings *s, int n_channels, const double *freq_center_per_channel, int device, jaero_batch **out)
{
    BatchPlan plan;
    const char *bad = out ? batch_plan(s, n_channels, plan) : "jaero_batch_create: bad argument";
    if (bad) { set_error(bad); return JAERO_E_ARG; }
    NewHandle<jaero_batch> nh(jaero_batch_destroy);
    int r = nh.open(device, "jaero_batch_create"); if (r) return r;
    jaero_batch *b = nh.h;
    HandleAllocs &A = b->allocs;
    cudaStream_t st = b->stream;
    b->own_stream = st;
    { const char *e = getenv("JAERO_OQPSK_PIPE"); b->use_pipe = !(e && e[0] == '0'); }
    DemodParams &p = b->p;
    p = plan.p;
    const size_t cp = p.cpad;
    int rc = 0;
    rc |= A.zeroed(&p.D, (size_t)D_COUNT * cp, st);
    rc |= A.zeroed(&p.I, (size_t)I_COUNT * cp, st);
    rc |= A.zeroed(&p.agc_ring, (size_t)p.agc_len * cp, st);
    if (p.report_ebno) { rc |= A.zeroed(&p.ebno_e1, (size_t)p.ebno_len * cp, st); rc |= A.zeroed(&p.ebno_e2, (size_t)p.ebno_len * cp, st); }
    rc |= A.zeroed(&p.fir_re, (size_t)(p.ntaps + 1) * cp, st);
    rc |= A.zeroed(&p.fir_im, (size_t)(p.ntaps + 1) * cp, st);
    {
        // The coarse estimate of a trigger is only consumed by channels that are unlocked, have no carrier detect or are about
        // to re-centre (FreqOffsetEstimateSlot, oqpskdemodulator.cpp:629-677), so in steady state the estimator kernels can run
        // on a second stream while the next segment is demodulated. Conditions: the warp-specialised 10500 bps kernel, the
        // non-cpuReduce schedule, and a segment grid that is fully resident (a waiting CTA must never keep the estimator's
        // CTAs from being scheduled). OFF unless JAERO_ASYNC_CFE=1: measured on B200 (4096 channels) the estimator's FP64 work,
        // when it shares SMs with the latency-bound segment warps, slows both kernels by 3-4x (FP64 pipe contention).
        cudaDeviceProp prop;
        JB_CUDA(cudaGetDeviceProperties(&prop, device));
        const char *e = getenv("JAERO_ASYNC_CFE");
        const int grid = (n_channels + 31) / 32;
        b->async_cfe = (e && e[0] == '1') && s->kind == JAERO_KIND_OQPSK && s->fb != 8400 && !s->cpu_reduce && b->use_pipe &&
                       grid <= prop.multiProcessorCount;
        p.bb_len = b->async_cfe ? p.bbnfft + p.bbnfft / 4 : p.bbnfft;
        if (b->async_cfe) {
            JB_CUDA(cudaStreamCreateWithFlags(&b->cfe_stream, cudaStreamNonBlocking));
            JB_CUDA(cudaEventCreateWithFlags(&b->ev_seg_done, cudaEventDisableTiming));
            JB_CUDA(cudaEventCreateWithFlags(&b->ev_cfe_done[0], cudaEventDisableTiming));
            JB_CUDA(cudaEventCreateWithFlags(&b->ev_cfe_done[1], cudaEventDisableTiming));
        }
        rc |= A.zeroed(&p.cfe_flag, (size_t)1, st);
    }
    rc |= A.zeroed(&p.bb, (size_t)n_channels * p.bb_len, st);
    rc |= A.zeroed(&p.marg_ring, (size_t)p.marg_len * cp, st);
    rc |= A.zeroed(&p.mse_pm, (size_t)p.mse_len * cp, st);
    rc |= A.zeroed(&p.mse_ma, (size_t)p.mse_len * cp, st);
    rc |= A.zeroed(&p.dt_ring, (size_t)p.dt_len * cp, st);
    if (s->kind == JAERO_KIND_MSK) {
        rc |= A.zeroed(&p.dsmpl_ring, (size_t)(p.sps + 1) * cp, st);
        rc |= A.zeroed(&p.dly8_ring, (size_t)(p.sps / 2 + 1) * cp, st);
    }
    rc |= A.zeroed(&p.soft, (size_t)n_channels * p.soft_cap, st);
    rc |= A.zeroed(&p.soft_total, (size_t)cp, st);
    rc |= A.zeroed(&p.lost_pos, (size_t)LOST_CAP * cp, st);
    rc |= A.zeroed(&p.cfe_est_out, (size_t)cp, st);
    {
        std::vector<double> sn, cs;
        trig_tables(sn, cs);
        double *ds = 0, *dc = 0;
        rc |= A.upload(&ds, sn, st); rc |= A.upload(&dc, cs, st);
        p.sin_t = ds; p.cos_t = dc;
    }
    // coarse estimator (CoarseFreqEstimate::setSettings, coarsefreqestimate.cpp:39-76)
    CfePlan &c = b->cfe;
    c = plan.cfe;
    // channels per pass group: the two work buffers of a group (2 x group x nfft x 16 B) (larger groups amortise launch tails; measured best at >= 512 on B200)
    int grp = 1024;
    if (const char *e = getenv("JAERO_CFE_GROUP")) grp = std::max(1, atoi(e));
    c.group = std::min(n_channels, grp);
    if (c.nfft == 16384) {
        const char *e = getenv("JAERO_CFE_CLUSTER");
        if (!(e && e[0] == '0')) c.clusters = cfe_cluster_capacity();
    }
    rc |= A.upload(&c.tw, plan.cfe_tw, st);
    rc |= A.zeroed(&c.work_a, (size_t)c.group * c.nfft, st); rc |= A.zeroed(&c.work_b, (size_t)c.group * c.nfft, st);
    rc |= A.zeroed(&c.y, (size_t)n_channels * c.nfft, st);
    if (c.is8400) rc |= A.upload(&c.window, plan.cfe_window, st);
    if (!plan.pre_H.empty()) {
        // K6: 2049-tap RRC (alpha 0.6) applied by streaming FFT convolution, nfft 4096 (oqpskdemodulator.cpp:280-283)
        b->pre_on = true;
        FirStream &f = b->fir;
        PreParams &q = b->pre;
        rc |= A.upload(&f.H, plan.pre_H, st); rc |= A.upload(&f.tw, plan.pre_tw, st);
        rc |= A.zeroed(&f.hist, (size_t)n_channels * FIR_L, st); rc |= A.zeroed(&f.inblk, (size_t)n_channels * FIR_L, st);
        rc |= A.zeroed(&f.outblk, (size_t)n_channels * FIR_L, st);
        rc |= A.zeroed(&p.m2_freq_sum, (size_t)cp, st);
        // mixer_fir_pre.SetFreq(freq_center,Fs) is only done in the ctor, with the ctor's 8000 Hz (oqpskdemodulator.cpp:21,115)
        std::vector<double> osc(4 * cp, 0.0);
        for (size_t c2 = 0; c2 < cp; c2++) { osc[1 * cp + c2] = (8000.0) * ((double)jb::WTSIZE) / ((double)((float)48000)); osc[2 * cp + c2] = 8000.0; }
        rc |= A.upload(&q.osc, osc, st);
        q.n_channels = n_channels; q.cpad = p.cpad; q.sin_t = p.sin_t; q.cos_t = p.cos_t;
    }
    // per-channel initial state
    std::vector<double> fc(n_channels);
    for (int i = 0; i < n_channels; i++) fc[i] = freq_center_per_channel ? freq_center_per_channel[i] : s->freq_center;
    double *dfc = 0;
    rc |= A.upload(&dfc, fc, st);
    if (rc) return JAERO_E_CUDA;
    init_state_kernel<<<(n_channels + 127) / 128, 128, 0, st>>>(p, dfc, plan.st_freq, 0.0);
    JB_CUDA(cudaGetLastError());
    if (s->kind == JAERO_KIND_OQPSK && s->fb > 8400 && b->use_pipe && !s->cpu_reduce) {
        // the pipelined kernel seats channels by symbol-timing phase: first after 2.9 s of signal (the timing loops' phases are final
        // to a few hundredths of a sample by then; at 2 s they are not), a check 2.7 s later (a no-op unless they moved),
        // then every JAERO_REGROUP_EPOCHS estimator epochs (default 128 = 11 s; 0 = never: symbol clocks of different transmitters
        // drift by a sample in minutes, not seconds)
        const char *e = getenv("JAERO_REGROUP_EPOCHS");
        b->regroup_every = e ? atoi(e) : 128;
        b->slot_of.resize(cp);
        std::vector<int> ident(2 * cp, 0);
        for (size_t c = 0; c < cp; c++) { ident[c] = (int)c; b->slot_of[c] = (int)c; }
        if (A.upload(&b->d_chan_of, ident, st) || A.zeroed(&b->d_keys, (size_t)cp, st) || A.pinned(&b->h_keys, cp)) return JAERO_E_CUDA;
        p.chan_of = b->d_chan_of;
        b->next_regroup = b->regroup_every > 0 ? 34 : -1;
    }
    if (A.pinned(&b->h_ints, (size_t)I_COUNT * cp) || A.pinned(&b->h_dbls, (size_t)D_COUNT * cp) || A.pinned(&b->h_soft_total, cp) ||
        A.pinned(&b->h_soft_stage, (size_t)n_channels * p.soft_cap)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(st));
    *out = nh.release();
    return JAERO_OK;
}

void jaero_batch_destroy(jaero_batch *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    cudaStreamSynchronize(b->stream);
    if (b->cfe_stream) { cudaStreamSynchronize(b->cfe_stream); cudaStreamDestroy(b->cfe_stream); }
    if (b->copy_stream) { cudaStreamSynchronize(b->copy_stream); cudaStreamDestroy(b->copy_stream); }
    if (b->ev_stage_free) cudaEventDestroy(b->ev_stage_free);
    for (int k = 0; k < 8; k++) if (b->ev_slice[k]) cudaEventDestroy(b->ev_slice[k]);
    if (b->ev_seg_done) cudaEventDestroy(b->ev_seg_done);
    for (int k = 0; k < 2; k++) if (b->ev_cfe_done[k]) cudaEventDestroy(b->ev_cfe_done[k]);
    for (auto &e : b->ev_seg) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    for (auto &e : b->ev_cfe) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    b->allocs.free_all(); b->stage.release(); b->x.release();
    if (b->own_stream) cudaStreamDestroy(b->own_stream);
    delete b;
}
int jaero_batch_channels(const jaero_batch *b) { return b ? b->p.n_channels : 0; }
int64_t jaero_batch_launch_count(const jaero_batch *b) { return b ? b->launches : 0; }

int jaero_batch_set_stream(jaero_batch *b, void *cuda_stream)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    b->stream = cuda_stream ? (cudaStream_t)cuda_stream : b->own_stream;
    return JAERO_OK;
}
int jaero_batch_set_profiling(jaero_batch *b, int enabled)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    b->profiling = enabled != 0;
    return JAERO_OK;
}
int jaero_batch_get_profile(jaero_batch *b, double out[5])
{
    if (!b || !out) { set_error("null argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    double seg = 0, cfe = 0;
    for (auto &e : b->ev_seg) { float ms = 0; cudaEventElapsedTime(&ms, e.first, e.second); seg += ms; cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    for (auto &e : b->ev_cfe) { float ms = 0; cudaEventElapsedTime(&ms, e.first, e.second); cfe += ms; cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    out[0] = seg; out[1] = (double)b->ev_seg.size(); out[2] = cfe; out[3] = (double)b->ev_cfe.size(); out[4] = b->prof_samples;
    b->ev_seg.clear(); b->ev_cfe.clear(); b->prof_samples = 0;
    return JAERO_OK;
}
int jaero_batch_sync(jaero_batch *b)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    return JAERO_OK;
}

int jaero_batch_write_device(jaero_batch *b, const int16_t *d_pcm, size_t n, size_t stride)
{
    if (!b || !d_pcm) { set_error("jaero_batch_write_device: null argument"); return JAERO_E_ARG; }
    if (n == 0) return JAERO_OK;                                   // `if(!len)return 0;` oqpskdemodulator.cpp:337
    if (stride < n || n > 0x7fffffff) { set_error("jaero_batch_write_device: bad stride / length"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const DemodParams &p = b->p;
    if ((((uintptr_t)d_pcm) & 15) || (stride & 7)) {
        // the kernels stage PCM rows with 16-byte bulk copies: re-pitch unaligned caller buffers on the device
        const size_t C = p.n_channels, pitch = (n + 7) & ~(size_t)7;
        if (d_pcm == b->stage.ptr) { set_error("internal: staging buffer misaligned"); return JAERO_E_STATE; }
        if (b->stage.reserve(C * pitch, b->stream)) return JAERO_E_CUDA;
        JB_CUDA(cudaMemcpy2DAsync(b->stage.ptr, pitch * sizeof(int16_t), d_pcm, stride * sizeof(int16_t), n * sizeof(int16_t), C,
                                  cudaMemcpyDeviceToDevice, b->stream));
        d_pcm = b->stage.ptr; stride = pitch;
    }
    if (b->pre_on) {
        while (b->next_slice < b->n_slices) { JB_CUDA(cudaStreamWaitEvent(b->stream, b->ev_slice[b->next_slice], 0)); b->next_slice++; }
        // K6 over the whole call first (oqpskdemodulator.cpp:343-381), then the per-sample loop consumes its output
        const size_t C = p.n_channels, xs = (n + 7) & ~(size_t)7;
        if (b->x.reserve(C * xs, b->stream)) return JAERO_E_CUDA;
        b->pre.x = b->x.ptr; b->pre.xstride = xs;
        b->p.xpre = b->x.ptr; b->p.xstride = xs;
        if (pre_down_launch(b->pre, d_pcm, stride, (int)n, b->stream)) return JAERO_E_CUDA;
        b->launches++;
        int i = 0;
        while (i < (int)n) {
            const int room = FIR_L - b->fir_fill;
            const int take = std::min(room, (int)n - i);
            if (fir_exchange_up_launch(b->pre, b->fir, i, i + take, b->fir_fill, b->stream)) return JAERO_E_CUDA;
            b->launches++;
            b->fir_fill += take; i += take;
            if (b->fir_fill == FIR_L) {
                if (fir_block_launch(b->fir, p.n_channels, b->fir_blocks == 0 ? 1 : 0, b->stream)) return JAERO_E_CUDA;
                b->launches++;
                b->fir_fill = 0; b->fir_blocks++;
            }
        }
    }
    peak_kernel<<<(p.n_channels + 3) / 4, 128, 0, b->stream>>>(p, d_pcm, stride, (int)n);
    JB_CUDA(cudaGetLastError());
    b->launches++;
    const int N = p.bbnfft;
    SegmentArgs a;
    memset(&a, 0, sizeof a);
    a.new_write = 1;
    int seg_start = 0; bool resume = false;
    auto launch = [&](int i0, int i1, bool stop_after_a, int bb0, int cc0) -> int {
        a.sample0 = b->samples; a.i0 = i0; a.i1 = i1; a.skip_a_first = resume ? 1 : 0; a.stop_after_a = stop_after_a ? 1 : 0;
        a.apply_cfe = resume ? 1 : 0; a.bb_pos = bb0; a.coarse_counter = cc0;
        a.cfe_wait = (resume && b->async_cfe) ? b->cfe_count : 0;
        while (b->next_slice < b->n_slices && b->next_slice * b->slice_len < i1) {   // input slices this segment reads
            JB_CUDA(cudaStreamWaitEvent(b->stream, b->ev_slice[b->next_slice], 0));
            b->next_slice++;
        }
        long long *d_trace = 0;
        if (const char *tf = getenv("JAERO_PIPE_TRACE")) {   // development aid: stage time stamps of one K1a launch
            if (!b->trace_state && b->launches > 300 && (i1 - i0) > 4000 && p.kind == JAERO_KIND_OQPSK && b->use_pipe && !p.xpre && p.fb > 8400) {
                (void)tf; cudaMalloc(&d_trace, 64 * 16 * sizeof(long long)); cudaMemset(d_trace, 0, 64 * 16 * sizeof(long long));
                a.trace = d_trace; a.trace_j0 = 2000;
            }
        }
        cudaEvent_t e0 = 0, e1 = 0;
        if (b->profiling) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, b->stream); }
        int r = (p.kind == JAERO_KIND_OQPSK) ? ((b->use_pipe && !p.xpre && p.fb > 8400) ? oqpsk_pipe_launch(p, a, d_pcm, stride, b->stream)
                                                                          : oqpsk_segment_launch(p, a, d_pcm, stride, b->stream))
                                             : ((b->use_pipe && (p.agc_len % 32) == 0 && (p.ebno_len % 32) == 0) ? msk_pipe_launch(p, a, d_pcm, stride, b->stream)
                                                                                                                      : msk_segment_launch(p, a, d_pcm, stride, b->stream));
        if (b->profiling) { cudaEventRecord(e1, b->stream); b->ev_seg.push_back({e0, e1}); b->prof_samples += (i1 - i0 - (stop_after_a ? 1 : 0)); }
        if (d_trace) {
            std::vector<long long> h(64 * 16);
            cudaStreamSynchronize(b->stream);
            cudaMemcpy(h.data(), d_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
            if (FILE *f = fopen(getenv("JAERO_PIPE_TRACE"), "w")) {
                for (int jj = 0; jj < 64; jj++) { for (int k = 0; k < 16; k++) fprintf(f, "%lld ", h[jj * 16 + k]); fprintf(f, "\n"); }
                fclose(f);
            }
            cudaFree(d_trace); a.trace = 0; b->trace_state = 1;
        }
        b->launches++;
        a.new_write = 0;
        return r;
    };
    TriggerSchedule &t = b->trig;
    int seg_bb = t.phys, seg_cc = t.cc;                            // counters at the start of the open segment
    bool cfe_in_flight = false;
    for (int i = 0; i < (int)n; i++) {
        // A(i): ring write + trigger test (oqpskdemodulator.cpp:410-429) — lock-step for the whole batch
        if (t.step(p)) {
            if (launch(seg_start, i + 1, true, seg_bb, seg_cc)) return JAERO_E_CUDA;
            b->samples += (i - seg_start);                         // samples whose B part has run
            cudaEvent_t c0 = 0, c1 = 0;
            int oldest = t.phys + (p.bb_len - N); if (oldest >= p.bb_len) oldest -= p.bb_len;
            cudaStream_t cs = b->async_cfe ? b->cfe_stream : b->stream;
            if (b->async_cfe) {
                JB_CUDA(cudaEventRecord(b->ev_seg_done, b->stream));
                JB_CUDA(cudaStreamWaitEvent(cs, b->ev_seg_done, 0));
            }
            if (b->profiling) { cudaEventCreate(&c0); cudaEventCreate(&c1); cudaEventRecord(c0, cs); }
            if (b->cfe.clusters > 0 ? cfe_cluster_run(b->cfe, p, oldest, std::min(b->cfe.clusters, p.n_channels), cs, &b->launches)
                                    : cfe_run(b->cfe, p, oldest, cs, &b->launches)) return JAERO_E_CUDA;
            if (b->profiling) { cudaEventRecord(c1, cs); b->ev_cfe.push_back({c0, c1}); }
            if (b->async_cfe) {
                b->cfe_count++;
                if (cfe_mark_launch(p.cfe_flag, b->cfe_count, cs)) return JAERO_E_CUDA;
                b->launches++;
                JB_CUDA(cudaEventRecord(b->ev_cfe_done[b->cfe_count & 1], cs));
                // the segment after the next one overwrites the quarter this estimate reads first: order the NEXT segment
                // behind the PREVIOUS estimate (a no-op in steady state)
                if (cfe_in_flight) JB_CUDA(cudaStreamWaitEvent(b->stream, b->ev_cfe_done[(b->cfe_count - 1) & 1], 0));
                cfe_in_flight = true;
            }
            b->epochs++;
            // seating check between two launches (the segment kernel has written its ring tiles back; per-channel state is indexed
            // by channel, only the ring rows and chan_of move)
            if (b->regroup_every > 0 && b->next_regroup >= 0 && b->epochs >= b->next_regroup) {
                if (batch_regroup_by_phase(b, false)) return JAERO_E_CUDA;
                b->next_regroup = b->epochs + (b->epochs < 64 ? std::min(32, b->regroup_every) : b->regroup_every);
            }
            seg_start = i; resume = true; seg_bb = t.phys; seg_cc = 0;
        }
    }
    if (launch(seg_start, (int)n, false, seg_bb, seg_cc)) return JAERO_E_CUDA;
    b->samples += ((int)n - seg_start);
    while (b->next_slice < b->n_slices) { JB_CUDA(cudaStreamWaitEvent(b->stream, b->ev_slice[b->next_slice], 0)); b->next_slice++; }
    b->n_slices = 0; b->next_slice = 0;
    if (cfe_in_flight) JB_CUDA(cudaStreamWaitEvent(b->stream, b->ev_cfe_done[b->cfe_count & 1], 0));   // join: a call leaves nothing in flight
    if (b->pre_on) {                                               // :608 mixer_fir_pre.SetFreq(mixer2_freq_sum/i)
        if (pre_finish_launch(b->pre, p.m2_freq_sum, (int)n, p.Fs, b->stream)) return JAERO_E_CUDA;
        b->launches++;
    }
    return JAERO_OK;
}

int jaero_batch_write(jaero_batch *b, const int16_t *pcm, size_t n, size_t stride)
{
    if (!b || !pcm) { set_error("jaero_batch_write: null argument"); return JAERO_E_ARG; }
    if (n == 0) return JAERO_OK;
    if (stride < n) { set_error("jaero_batch_write: channel_stride < n_samples"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const size_t C = b->p.n_channels;
    const size_t pitch = (n + 7) & ~(size_t)7;
    if (b->stage.reserve(C * pitch, b->stream)) return JAERO_E_CUDA;
    if (n < 8192) {
        JB_CUDA(cudaMemcpy2DAsync(b->stage.ptr, pitch * sizeof(int16_t), pcm, stride * sizeof(int16_t), n * sizeof(int16_t), C,
                                  cudaMemcpyHostToDevice, b->stream));
        return jaero_batch_write_device(b, b->stage.ptr, n, pitch);
    }
    // long calls: copy in column slices on a second stream so that the transfer of later samples overlaps the
    // demodulation of earlier ones (pinned host memory makes the copies truly asynchronous)
    if (!b->copy_stream) {
        JB_CUDA(cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking));
        JB_CUDA(cudaEventCreateWithFlags(&b->ev_stage_free, cudaEventDisableTiming));
        for (int k = 0; k < 8; k++) JB_CUDA(cudaEventCreateWithFlags(&b->ev_slice[k], cudaEventDisableTiming));
    }
    JB_CUDA(cudaEventRecord(b->ev_stage_free, b->stream));          // everything already queued that reads the staging buffer
    JB_CUDA(cudaStreamWaitEvent(b->copy_stream, b->ev_stage_free, 0));
    b->slice_len = (int)((((n + 7) / 8) + 7) & ~(size_t)7);
    b->n_slices = 0; b->next_slice = 0;
    for (size_t s0 = 0; s0 < n; s0 += (size_t)b->slice_len) {
        const size_t len = std::min((size_t)b->slice_len, n - s0);
        JB_CUDA(cudaMemcpy2DAsync(b->stage.ptr + s0, pitch * sizeof(int16_t), pcm + s0, stride * sizeof(int16_t), len * sizeof(int16_t), C,
                                  cudaMemcpyHostToDevice, b->copy_stream));
        JB_CUDA(cudaEventRecord(b->ev_slice[b->n_slices], b->copy_stream));
        b->n_slices++;
    }
    return jaero_batch_write_device(b, b->stage.ptr, n, pitch);
}

static int pull_ints(jaero_batch *b)
{
    const size_t cp = b->p.cpad;
    JB_CUDA(cudaMemcpyAsync(b->h_ints, b->p.I, (size_t)I_COUNT * cp * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    JB_CUDA(cudaStreamSynchronize(b->stream));
    return 0;
}

int jaero_batch_read_softbits(jaero_batch *b, int16_t *out, size_t cap, int32_t *counts)
{
    if (!b || !out || !counts) { set_error("jaero_batch_read_softbits: null argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    if (pull_ints(b)) return JAERO_E_CUDA;
    const DemodParams &p = b->p;
    const size_t cp = p.cpad;
    const int *cnt = b->h_ints + (size_t)I_SOFT_COUNT * cp, *ovf = b->h_ints + (size_t)I_SOFT_OVERFLOW * cp;
    const int r = read_soft_rows(cnt, ovf, p.n_channels, p.soft, p.soft_cap, b->h_soft_stage, out, cap, counts, b->stream);
    return r ? r : batch_soft_reset(b, b->stream);
}
int jaero_batch_softbits_device(jaero_batch *b, const int16_t **d_soft, const int32_t **d_counts, size_t *ring_cap)
{
    if (!b || !d_soft || !d_counts || !ring_cap) { set_error("null argument"); return JAERO_E_ARG; }
    *d_soft = b->p.soft; *d_counts = b->p.I + (size_t)I_SOFT_COUNT * b->p.cpad; *ring_cap = (size_t)b->p.soft_cap;
    return JAERO_OK;
}
int jaero_batch_reset_softbits(jaero_batch *b)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    return batch_soft_reset(b, b->stream);
}
int jaero_batch_set_dcd(jaero_batch *b, int channel, int dcd)
{
    if (!b || channel >= b->p.n_channels) { set_error("jaero_batch_set_dcd: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    set_int_kernel<<<(b->p.n_channels + 127) / 128, 128, 0, b->stream>>>(b->p, I_DCD, channel, dcd ? 1 : 0);
    JB_CUDA(cudaGetLastError());
    return JAERO_OK;
}
int jaero_batch_set_center_freq(jaero_batch *b, int channel, double hz)
{
    if (!b || channel >= b->p.n_channels) { set_error("jaero_batch_set_center_freq: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    center_freq_kernel<<<(b->p.n_channels + 127) / 128, 128, 0, b->stream>>>(b->p, channel, hz);
    JB_CUDA(cudaGetLastError());
    return JAERO_OK;
}
// setAFC / setSQL / setCPUReduce (oqpskdemodulator.cpp:149-167, mskdemodulator.cpp:113-131): plain flags the sample loop reads;
// the kernels take them by value at every launch, so a change applies from the next write on
int jaero_batch_set_afc(jaero_batch *b, int state)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    b->p.afc = state ? 1 : 0;
    return JAERO_OK;
}
int jaero_batch_set_sql(jaero_batch *b, int state)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    b->p.sql = state ? 1 : 0;
    return JAERO_OK;
}
// connect(demodulator, SignalStatus(bool), aerol, SignalStatusSlot(bool)) (JAERO/mainwindow.cpp:432,508)
int jaero_batch_wire_signal_status(jaero_batch *b, int enabled)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    b->p.wire_sigstat = enabled ? 1 : 0;
    return JAERO_OK;
}
// Seat the channels of the pipelined 10500 bps kernel: slot_of[c] = seat of channel c (a permutation of 0..n_channels-1), or NULL
// to seat them by symbol-timing phase now. Results never depend on the seating (channels do not interact); throughput does.
int jaero_batch_regroup(jaero_batch *b, const int32_t *slot_of)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    if (!b->d_chan_of) return JAERO_OK;                        // this batch's kernel has a fixed seating
    JB_CUDA(cudaSetDevice(b->device));
    if (!slot_of) return batch_regroup_by_phase(b, true) ? JAERO_E_CUDA : JAERO_OK;
    const int C = b->p.n_channels, cp = b->p.cpad;
    std::vector<int> v(cp), seen(C, 0);
    for (int c = 0; c < C; c++) { if (slot_of[c] < 0 || slot_of[c] >= C || seen[slot_of[c]]) { set_error("jaero_batch_regroup: not a permutation"); return JAERO_E_ARG; } seen[slot_of[c]] = 1; v[c] = slot_of[c]; }
    for (int c = C; c < cp; c++) v[c] = c;
    return batch_apply_seating(b, v) ? JAERO_E_CUDA : JAERO_OK;
}
int jaero_batch_set_cpu_reduce(jaero_batch *b, int state)
{
    if (!b) { set_error("null handle"); return JAERO_E_ARG; }
    if (b->async_cfe) { set_error("jaero_batch_set_cpu_reduce: not available with JAERO_ASYNC_CFE=1"); return JAERO_E_STATE; }
    b->p.cpu_reduce = state ? 1 : 0;
    return JAERO_OK;
}
int jaero_batch_get_status_all(jaero_batch *b, jaero_status *out)
{
    if (!b || !out) { set_error("null argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(b->device));
    const size_t cp = b->p.cpad;
    JB_CUDA(cudaMemcpyAsync(b->h_dbls, b->p.D, (size_t)D_COUNT * cp * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
    JB_CUDA(cudaMemcpyAsync(b->h_soft_total, b->p.soft_total, cp * sizeof(long long), cudaMemcpyDeviceToHost, b->stream));
    if (pull_ints(b)) return JAERO_E_CUDA;
    for (int ch = 0; ch < b->p.n_channels; ch++) {
        auto D = [&](int i) { return b->h_dbls[(size_t)i * cp + ch]; };
        auto I = [&](int i) { return b->h_ints[(size_t)i * cp + ch]; };
        jaero_status &s = out[ch];
        s.mixer2_freq = D(D_M2_FREQ); s.mixer2_wtptr = D(D_M2_PTR); s.center_freq = D(D_MC_FREQ);
        s.st_freq = D(D_ST_FREQ); s.st_wtptr = D(D_ST_PTR); s.agc = D(D_AGC_VAL); s.mse = D(D_MSE);
        s.ebno = D(D_EB_EBNO); s.marg = D(D_MARG_VAL); s.cfe_est = D(D_CFE_EST);
        s.n_sig_true = I(I_SIG_TRUE); s.n_sig_false = I(I_SIG_FALSE);
        s.center_wtptr = D(D_MC_PTR); s.st_ref_wtptr = D(D_SR_PTR);
        s.samples = b->samples; s.softbits = b->h_soft_total[ch] + I(I_SOFT_COUNT); s.dcd = I(I_DCD); s.reserved = 0;
        s.peak_volume = (double)I(I_PEAK) / 32768.0;
        s.scatter[0] = D(D_SCAT0_RE); s.scatter[1] = D(D_SCAT0_IM); s.scatter[2] = D(D_SCAT1_RE); s.scatter[3] = D(D_SCAT1_IM);
    }
    // `emit PeakVolume(maxval); maxval=0;`: the read-out restarts the maximum
    JB_CUDA(cudaMemsetAsync(b->p.I + (size_t)I_PEAK * cp, 0, cp * sizeof(int), b->stream));
    return JAERO_OK;
}
int jaero_batch_get_status(jaero_batch *b, int channel, jaero_status *out)
{
    if (!b || !out || channel < 0 || channel >= b->p.n_channels) { set_error("jaero_batch_get_status: bad argument"); return JAERO_E_ARG; }
    std::vector<jaero_status> all(b->p.n_channels);
    int r = jaero_batch_get_status_all(b, all.data());
    if (r) return r;
    *out = all[channel];
    return JAERO_OK;
}

} // extern "C"
