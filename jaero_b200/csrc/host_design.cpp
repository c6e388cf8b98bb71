// Host-side design math of the handles (see host_design.h). Compiled with the library's host flags (-O3 -fno-fast-math).
#include "host_design.h"
#include <algorithm>
#include <cmath>
#include <cstring>

namespace jb {

std::vector<double> rrc_taps(double alpha, int firsize, double samplerate, double symbol_freq)
{
    if ((firsize % 2) == 0) firsize += 1;
    std::vector<double> pts(firsize);
    const double T = (samplerate) / (symbol_freq);
    for (int i = 0; i < firsize; i++) {
        if (i == ((firsize - 1) / 2)) pts[i] = (4.0 * alpha + M_PI - M_PI * alpha) / (M_PI * sqrt(T));
        else {
            const double fi = (((double)i) - ((double)(firsize - 1)) / 2.0);
            if (fabs(1.0 - pow(4.0 * alpha * fi / T, 2)) < 0.0000000001)
                pts[i] = (alpha * ((M_PI - 2.0) * cos(M_PI / (4.0 * alpha)) + (M_PI + 2.0) * sin(M_PI / (4.0 * alpha))) / (M_PI * sqrt(2.0 * T)));
            else
                pts[i] = (4.0 * alpha / (M_PI * sqrt(T)) * (cos((1.0 + alpha) * M_PI * fi / T) + T / (4.0 * alpha * fi) * sin((1.0 - alpha) * M_PI * fi / T)) / (1.0 - pow(4.0 * alpha * fi / T, 2)));
        }
    }
    return pts;
}

bool delay_weights(double fd, std::vector<double> &w)
{
    const int size = (int)std::ceil(fd) + 1;
    w.assign(std::max(size, 0), 0.0);
    bool shift = size >= 1;
    for (int bp = 0; bp < size; bp++) {
        double dptr = ((double)bp) - fd;
        while (std::floor(dptr) < 0) dptr += ((double)size);
        const int iptr = (int)std::floor(dptr);
        w[bp] = dptr - ((double)iptr);
        int expect = bp - (int)std::ceil(fd); while (expect < 0) expect += size;
        if (iptr != expect) shift = false;
    }
    return shift;
}

cvec twiddles(int n)
{
    cvec tw(n);
    for (int k = 0; k < n; k++) { const double a = -2.0 * M_PI * (double)k / (double)n; tw[k] = std::complex<double>(cos(a), sin(a)); }
    return tw;
}

void fft_radix2(cvec &x, const cvec &tw)
{
    const int NF = (int)x.size();
    int bits = 0;
    while ((1 << bits) < NF) bits++;
    for (int i = 0; i < NF; i++) { int r = 0; for (int q = 0; q < bits; q++) if (i & (1 << q)) r |= 1 << (bits - 1 - q); if (r > i) std::swap(x[i], x[r]); }
    for (int len = 2; len <= NF; len <<= 1)
        for (int i = 0; i < NF; i += len)
            for (int k = 0; k < len / 2; k++) { auto w = tw[k * (NF / len)]; auto u = x[i + k], v = x[i + k + len / 2] * w; x[i + k] = u + v; x[i + k + len / 2] = u - v; }
}

void trig_tables(std::vector<double> &sn, std::vector<double> &cs)
{
    sn.resize(WTSIZE); cs.resize(WTSIZE);
    for (int i = 0; i < WTSIZE; i++) sn[i] = (sin(2 * M_PI * ((double)i) / WTSIZE));
    for (int i = 0; i < WTSIZE; i++) cs[i] = (sin(M_PI_2 + 2 * M_PI * ((double)i) / WTSIZE));
}

std::vector<uint8_t> scrambler_sequence(int n)
{
    int st[15] = {1, 1, 0, 1, 0, 0, 1, 0, 1, 0, 1, 1, 0, 0, 1};
    std::vector<uint8_t> seq(n);
    for (int a = 0; a < n; a++) { const int v = st[0] ^ st[14]; seq[a] = (uint8_t)v; for (int i = 14; i > 0; i--) st[i] = st[i - 1]; st[0] = v; }
    return seq;
}

std::vector<double> estimator_window(int nfft, int startbin)
{
    std::vector<double> win(nfft, 0.0);
    win[0] = 1;
    for (int i = 1; i <= startbin; i++) {
        double val = cos(M_PI_2 * ((double)i) / ((double)startbin)); val *= val;
        if ((nfft - i) < 0) break;
        if (i >= nfft) break;
        win[nfft - i] = val; win[i] = val;
    }
    return win;
}

// Delay<T> with at most 4 ring positions in the shift-register form: the weights go into the kernel parameter block
static bool delay_weights4(double fd, int *k_out, double *w_out /*[4]*/)
{
    std::vector<double> w;
    const int size = (int)std::ceil(fd) + 1;
    if (size > 4 || size < 2 || !delay_weights(fd, w)) return false;
    for (int bp = 0; bp < size; bp++) w_out[bp] = w[bp];
    *k_out = (int)std::ceil(fd);
    return true;
}

const char *batch_plan(const jaero_settings *s, int n_channels, BatchPlan &plan)
{
    if (!s || n_channels <= 0) return "jaero_batch_create: bad argument";
    if (s->kind != JAERO_KIND_OQPSK && s->kind != JAERO_KIND_MSK) return "jaero_batch_create: unknown kind";
    if (s->Fs <= 0 || s->fb <= 0 || s->coarsefreqest_fft_power < 10 || s->coarsefreqest_fft_power > 14)
        return "jaero_batch_create: Fs/fb must be positive and coarsefreqest_fft_power in 10..14";
    DemodParams &p = plan.p;
    memset(&p, 0, sizeof p);
    p.kind = s->kind; p.n_channels = n_channels; p.cpad = (n_channels + 31) & ~31;
    p.Fs = s->Fs; p.fb = s->fb; p.lockingbw = s->lockingbw; p.signalthreshold = s->signalthreshold;
    p.afc = s->afc; p.sql = s->sql; p.cpu_reduce = s->cpu_reduce; p.report_ebno = s->report_ebno;
    p.bbnfft = 1 << s->coarsefreqest_fft_power;
    std::vector<double> taps;
    if (s->kind == JAERO_KIND_OQPSK) {
        taps = (s->fb == 8400) ? rrc_taps(0.6, 55, s->Fs, s->fb / 2) : rrc_taps(1.0, 55, s->Fs, s->fb / 2);   // oqpskdemodulator.cpp:209-211
        p.agc_len = (int)round(4 * s->Fs);                                    // :197 AGC(4,Fs)
        p.ebno_len = 2 * 48000;                                               // :42 (built in the ctor with Fs=48000)
        p.marg_len = 800; p.dt_len = 401; p.mse_len = 400;                    // :44-45,53
        const double T = s->Fs / (s->fb / 2);                                 // :221
        if (!delay_weights4(T / 4.0, &p.k41, p.w41v) || !delay_weights4(T / 8.0, &p.k8, p.w8v) || p.k41 > 3 || p.k8 > 3)
            return "unsupported fractional delay for this Fs/fb";
        if (s->fb == 8400) {                                                  // :243-250 (the 10 Hz set, assigned last, wins)
            p.res_b0 = 0.0012845857864470789; p.res_b1 = 0; p.res_b2 = -0.0012845857864470789;
            p.res_a1 = -0.90681461999279889; p.res_a2 = 0.99743082842710584;
            p.ee = 0.65;
        } else {
            p.res_b0 = 0.00032714218939589035; p.res_b1 = 0; p.res_b2 = 0.00032714218939589035;   // :256-261
            p.res_a1 = -0.39005299948210803; p.res_a2 = 0.99934571562120822;
            p.ee = 0.4;                                                       // :263
        }
        p.lf_b0 = 0.0010275610653672064; p.lf_b1 = 0.0020551221307344128; p.lf_b2 = 0.0010275610653672064;   // :95-100
        p.lf_a1 = -1.9207386815577139; p.lf_a2 = 0.92509247310306331;
        plan.st_freq = s->fb;                                                 // :270
    } else {
        p.sps = (int)(s->Fs / s->fb);                                         // mskdemodulator.cpp:149
        if (2 * p.sps > MAX_TAPS) return "MSK: 2*SamplesPerSymbol exceeds the supported FIR length";
        taps.resize(2 * p.sps);
        for (int i = 0; i < 2 * p.sps; i++) taps[i] = sin(M_PI * i / (2.0 * p.sps)) / (2.0 * p.sps);   // :164-170
        p.agc_len = (int)round(1 * s->Fs);                                    // :173
        p.ebno_len = (int)(2.0 * s->Fs);                                      // :176
        p.marg_len = p.sps; p.dt_len = p.sps / 2 + 1; p.mse_len = 600;        // :254-256, ctor :64
        if (s->fb >= 1200) {                                                  // :189-250
            p.correctionfactor = 0.6;
            if (s->Fs == 48000) { p.res_a1 = -1.993312819378528; p.res_a2 = 0.999476538254407; p.res_b0 = 2.617308727964618e-04; p.res_b2 = -2.617308727964618e-04; p.ee = 0.025; }
            else { p.res_a1 = -1.974342917561558; p.res_a2 = 0.998953350377616; p.res_b0 = 5.233248111921052e-04; p.res_b2 = -5.233248111921052e-04; p.ee = 0.05; }
        } else {
            p.correctionfactor = 1.0;
            if (s->Fs == 48000) { p.res_a1 = -1.998196509168551; p.res_a2 = 0.999738234875681; p.res_b0 = 1.308825621597620e-04; p.res_b2 = -1.308825621597620e-04; p.ee = 0.025; }
            else { p.res_a1 = -1.974342917561558; p.res_a2 = 0.998953350377616; p.res_b0 = 5.233248111921052e-04; p.res_b2 = -5.233248111921052e-04; p.ee = 0.0125; }
        }
        p.res_b1 = 0;
        plan.st_freq = s->fb / 2;                                             // :159
    }
    if ((p.agc_len % 32) || (p.ebno_len % 32) || p.agc_len < 96 || p.ebno_len < 96)
        return "unsupported sample rate: the AGC / EbNo window lengths must be multiples of 32 samples";
    p.ntaps = (int)taps.size();
    p.soft_cap = std::max(4096, (int)(2 * s->fb) + 64);
    if (p.ntaps > MAX_TAPS) return "too many FIR taps";
    for (int k = 0; k < p.ntaps; k++) p.taps[k] = taps[k];   // per-batch: the taps ride in the kernel parameter block

    // coarse estimator plan (CoarseFreqEstimate::setSettings, coarsefreqestimate.cpp:39-76)
    CfePlan &c = plan.cfe;
    memset(&c, 0, sizeof c);
    c.nfft = p.bbnfft;
    const int lg = s->coarsefreqest_fft_power;
    c.n1 = 1 << ((lg + 1) / 2); c.n2 = 1 << (lg / 2);
    c.hzperbin = s->Fs / ((double)c.nfft);
    const double lbw = (s->kind == JAERO_KIND_OQPSK) ? 2.0 * s->lockingbw / 2.0 : s->lockingbw;   // oqpskdemodulator.cpp:191
    c.startbin = (int)std::max(round(lbw / c.hzperbin), 1.0);
    c.stopbin = c.nfft - c.startbin;
    c.expectedpeakbin = (int)round(s->fb / (2.0 * c.hzperbin));
    c.lo = (int)round((-lbw / c.hzperbin) + ((double)(c.nfft / 2)));
    c.hi = (int)round((lbw / c.hzperbin) + ((double)(c.nfft / 2)));
    c.is8400 = (s->fb == 8400);
    plan.cfe_tw = twiddles(c.nfft);
    plan.cfe_window.clear();
    if (c.is8400) plan.cfe_window = estimator_window(c.nfft, c.startbin);
    plan.pre_H.clear(); plan.pre_tw.clear();
    if (s->kind == JAERO_KIND_OQPSK && s->fb == 8400) {
        // K6: 2049-tap RRC (alpha 0.6) applied by streaming FFT convolution, nfft 4096 (oqpskdemodulator.cpp:280-283)
        std::vector<double> kern = rrc_taps(0.6, 2048, s->Fs, s->fb / 2);
        const int NF = 4096;
        plan.pre_H.assign(NF, 0.0);
        for (size_t i = 0; i < kern.size(); i++) plan.pre_H[i] = kern[i];
        plan.pre_tw = twiddles(NF);
        fft_radix2(plan.pre_H, plan.pre_tw);
    }
    return nullptr;
}

const char *burst_plan(const jaero_settings *s, int n_channels, int kind, BurstPlan &plan)
{
    if (!s || n_channels <= 0) return "jaero_burst_create: bad argument";
    if (kind == 0 && (s->Fs != 48000 || (s->fb != 600 && s->fb != 1200))) return "jaero_burst_msk_create: burst MSK runs at Fs=48000 with fb 600 or 1200";
    if (kind == 1 && (s->Fs != 48000 || s->fb != 10500)) return "jaero_burst_oqpsk_create: burst OQPSK runs at Fs=48000, fb=10500";
    BurstParams &p = plan.p;
    memset(&p, 0, sizeof p);
    p.kind = kind; p.sql = s->sql;
    p.n_channels = n_channels; p.cpad = (n_channels + 31) & ~31;
    p.Fs = s->Fs; p.fb = s->fb; p.lockingbw = s->lockingbw; p.signalthreshold = s->signalthreshold; p.afc = 1;   // ctor: afc=true (:15)
    double fc = s->freq_center;
    if (fc > ((p.Fs / 2.0) - (p.lockingbw / 2.0))) fc = ((p.Fs / 2.0) - (p.lockingbw / 2.0));
    plan.freq_center = fc;
    p.sps = (int)(p.Fs / p.fb);
    const double SPS = kind == 1 ? 2.0 * p.Fs / p.fb : (double)p.sps;            // burstoqpskdemodulator.cpp:219
    p.spsd = SPS;
    std::vector<double> taps;
    if (kind == 1) { p.sps = (int)SPS; p.ntaps = 55; taps = rrc_taps(1.0, 55, 48000, 10500 / 2.0); }    // ctor :38-46
    else {
        p.ntaps = 2 * p.sps;
        if (p.ntaps > MAX_TAPS) return "burst MSK: matched filter too long";
        taps.resize(p.ntaps);
        for (int i = 0; i < p.ntaps; i++) taps[i] = sin(M_PI * i / (2.0 * SPS)) / (2.0 * SPS);      // :173-177
    }
    for (int k = 0; k < p.ntaps; k++) p.taps[k] = taps[k];
    p.agc_len = (int)round(1 * p.Fs);
    auto qround = [](double d) { return d >= 0.0 ? int(d + 0.5) : int(d - double(int(d - 1)) + 0.5) + int(d - 1); };
    double btdiff_fd = 0;
    if (kind == 1) {                                              // burstoqpskdemodulator.cpp:202-277
        p.btma_len = qround(128.0 * SPS); p.mav1_len = (int)(SPS * 128); btdiff_fd = SPS * 128; p.btdiff_len = (int)std::ceil(btdiff_fd) + 1;
        p.pd_len = (int)(SPS * 128.0 / 2.0); p.pd_threshold = 0.2;
        p.tri_sz = qround((256.0 + 16.0 + 16.0) * SPS); p.d1_len = (int)(SPS * 128.0 * 2.5 - 190) + 1; p.d2_len = p.tri_sz + 1;
        p.tri_nb = p.tri_nt = qround(128.0 * SPS);
        p.res_b0 = 0.0048847995518126464; p.res_b1 = 0; p.res_b2 = -0.0048847995518126464;       // ctor :69-75 (75 Hz)
        p.res_a1 = -0.3882746897971619; p.res_a2 = 0.99023040089637471;
        p.ee = 0.4;
    } else if (p.fb >= 1200) {                                           // :205-256
        p.btma_len = qround(126.0 * SPS); p.mav1_len = (int)(SPS * 126); p.btdiff_len = (int)std::ceil(SPS * 126) + 1;
        p.pd_len = (int)(SPS * 126.0 / 2.0); p.pd_threshold = 0.1;
        p.tri_sz = qround(200.0 * SPS); p.d1_len = ((int)289 * p.sps) + 20 + 1; p.d2_len = (int)(qround(72 + 120.0) * SPS) + 1;
        p.size_base = 126; p.size_top = 74; p.start_processing = 120; p.end_rotation = (int)((120 + 37) * SPS);
        p.res_a1 = -1.993312819378528; p.res_a2 = 0.999476538254407; p.res_b0 = 2.617308727964618e-04; p.res_b1 = 0; p.res_b2 = -2.617308727964618e-04;
        p.ee = 0.025; btdiff_fd = SPS * 126;
    } else {                                                      // :257-311
        p.btma_len = qround(150.0 * SPS); p.mav1_len = (int)(SPS * 150); p.btdiff_len = (int)std::ceil(SPS * 150) + 1;
        p.pd_len = (int)(SPS * 150.0 / 2.0); p.pd_threshold = 0.2;
        p.tri_sz = qround(224 * SPS); p.d1_len = ((int)397 * p.sps) + 20 + 1; p.d2_len = qround((72 + 150.0) * SPS) + 1;
        p.size_base = 150; p.size_top = 74; p.start_processing = 150; p.end_rotation = (int)((150 + 56) * SPS);
        p.res_a1 = -1.991228154418550; p.res_a2 = 0.997385427096603; p.res_b0 = 0.001307286451699; p.res_b1 = 0; p.res_b2 = -0.001307286451699;
        p.ee = 0.015; btdiff_fd = SPS * 150;
    }
    if (kind == 0) { p.tri_nb = (int)rint(p.size_base * SPS); p.tri_nt = (int)rint(p.size_top * SPS); }
    p.startstopstart = kind == 1 ? (int)(SPS * (1050)) : (int)(SPS * 500);
    p.btd1_len = (int)std::ceil(1.0 * SPS) + 1;
    if (!delay_weights(1.0 * SPS, plan.w_btd1) || !delay_weights(btdiff_fd, plan.w_btdiff) || !delay_weights(SPS / 2.0, plan.w_a1))
        return "burst: unsupported delay";
    p.a1_k = (int)std::ceil(SPS / 2.0);
    if (kind == 0) {
        // Delay<T> weight at ring position 0; the kernels take one weight, so it must be the same at every position
        std::vector<double> w8;
        delay_weights(SPS / 2.0, w8);
        for (double w : w8) if (w != w8[0]) return "burst MSK: unsupported delay";
        p.d8_k = (int)std::ceil(SPS / 2.0); p.d8_w = w8[0];
        p.eb_len = (int)(0.15 * p.Fs); p.agc2_len = (int)round((SPS * 128.0 / p.Fs) * p.Fs); p.ds_len = p.sps + 1; p.msema_len = 75;
    } else {
        const double sps0 = 2.0 * 48000 / 10500;                  // ctor :48-52
        if (!delay_weights4(sps0 / 4.0, &p.k41, p.w41v) || !delay_weights4(sps0 / 8.0, &p.k8, p.w8v)) return "burst OQPSK: unsupported delay";
        p.d8_k = 1; p.ds_len = 1;
        p.eb_len = (int)(SPS * (256.0)); p.agc2_len = (int)round((SPS * 64.0 / p.Fs) * p.Fs); p.msema_len = 128;
    }
    p.soft_cap = std::max(4096, (int)(2 * p.fb) + 64);
    p.astride = BURST_CHUNK;
    // Hilbert filter: QJHilbertFilter::setSize(2048) (DSP.cpp:759-789), streaming FFT convolution nfft 8192
    HilbertStream &h = plan.hil; memset(&h, 0, sizeof h);
    h.K = 2048; h.nfft = 8192; h.L = h.nfft - h.K + 1;
    const int N = h.K;
    plan.hil_H.assign(h.nfft, 0.0);
    for (int i = 0; i < N; i++) {
        if (i == N / 2) plan.hil_H[i] = std::complex<double>(-1, 0);
        else if ((i % 2) == 0) plan.hil_H[i] = 0;
        else plan.hil_H[i] = std::complex<double>(0, (2.0 / ((double)N)) / (std::tan(M_PI * (((double)i) / ((double)N) - 0.5))));
    }
    plan.hil_tw = twiddles(h.nfft);
    plan.tw32k = twiddles(TRI_N);
    fft_radix2(plan.hil_H, plan.hil_tw);
    return nullptr;
}

const char *pchannel_plan(int n_channels, double fb, PChanParams &pp)
{
    if (n_channels <= 0) return "jaero_pchannel_create: bad argument";
    const int ifb = (int)(fb + 0.5);
    if (ifb != 600 && ifb != 1200 && ifb != 10500) return "jaero_pchannel_create: P-channel rates are 600, 1200, 10500";
    memset(&pp, 0, sizeof pp);
    pp.n_channels = n_channels; pp.paddinglength = 24;                          // aerol.cpp:940
    switch (ifb) {                                                               // AeroL::setSettings, aerol.cpp:1013-1052
    case 600: pp.cols = 6; pp.number_of_bits = 1152; pp.bits_in_header = 16; pp.total_number_of_bits = 16 + 1152 + 32; pp.oqpsk = 0; pp.dl2_len = 576 - 6 + 1; break;
    case 1200: pp.cols = 9; pp.number_of_bits = 1152; pp.bits_in_header = 16; pp.total_number_of_bits = 16 + 1152 + 32; pp.oqpsk = 0; pp.dl2_len = 576 - 6 + 1; break;
    default: pp.cols = 78; pp.number_of_bits = 4992; pp.bits_in_header = 16 + 178; pp.total_number_of_bits = 16 + 178 + 4992 + 64; pp.oqpsk = 1; pp.dl2_len = 4992 - 6 + 1; break;
    }
    pp.block_len = pp.cols * 64;
    pp.info_cap = pp.number_of_bits / 16 + 16;
    // queue depth: a demodulator soft ring holds max(4096, 2*fb+64) values (batch_plan); a call may hand all of them over
    pp.queue = std::max(PCHAN_QUEUE_MIN, std::max(4096, 2 * ifb + 64) / pp.block_len + 2);
    pp.su_cap = pp.queue * (pp.number_of_bits / 2 / 96) + 8;
    return nullptr;
}

const char *rt_plan(double fb, int n_channels, RtParams &rp)
{
    if (n_channels <= 0) return "jaero_rt_create: bad argument";
    const int ifb = (int)(fb >= 0.0 ? fb + 0.5 : fb - 0.5);
    if (ifb != 600 && ifb != 1200 && ifb != 10500) return "jaero_rt_create: burst R/T channels run at 600, 1200 or 10500 bps";
    memset(&rp, 0, sizeof rp);
    rp.n_channels = n_channels; rp.ifb = ifb; rp.oqpsk = (ifb == 10500);
    rp.number_of_bits = (ifb == 10500) ? 4992 : 1152;                       // aerol.cpp:1012-1050
    rp.total_number_of_bits = rp.oqpsk ? ifb : ifb * 3;                     // :1062-1070
    return nullptr;
}

} // namespace jb
