// Text form of what a create call derives from its settings (kernel parameter blocks and host tables), one value per
// line, doubles as %.17g. tests/test_host_design_cpu.py hashes it per mode. Needs only the kernel parameter headers.
#pragma once
#include "../../jaero_b200/csrc/demod.cuh"
#include "../../jaero_b200/csrc/burst.cuh"
#include "../../jaero_b200/csrc/pchannel.cuh"
#include "../../jaero_b200/csrc/rtchannel.cuh"
#include <cstdio>

// settings of each mode the creates accept: {kind (0 OQPSK / 1 MSK), fft_power, freq_center, lockingbw, fb, Fs, signalthreshold}
struct PlanMode { const char *name; int burst; int kind; int fft_power; double fc, lockingbw, fb, Fs, thr; };
static const PlanMode PLAN_MODES[] = {
    {"oqpsk10500", 0, 0, 14, 8000.0, 10500.0, 10500.0, 48000.0, 0.65},
    {"oqpsk8400", 0, 0, 14, 8000.0, 8400.0, 8400.0, 48000.0, 0.65},
    {"msk600", 0, 1, 13, 1500.0, 1000.0, 600.0, 48000.0, 0.5},
    {"msk1200", 0, 1, 13, 1500.0, 1000.0, 1200.0, 48000.0, 0.5},
    {"burst_msk600", 1, 0, 13, 1500.0, 1000.0, 600.0, 48000.0, 0.5},
    {"burst_msk1200", 1, 0, 13, 1500.0, 1000.0, 1200.0, 48000.0, 0.5},
    {"burst_oqpsk10500", 1, 1, 14, 8000.0, 10500.0, 10500.0, 48000.0, 0.65},
};

static void dump_i(const char *k, long long v) { printf("%s %lld\n", k, v); }
static void dump_d(const char *k, double v) { printf("%s %.17g\n", k, v); }
static void dump_v(const char *k, const double *v, size_t n) { printf("%s %zu\n", k, n); for (size_t i = 0; i < n; i++) printf("%.17g\n", v[i]); }
static void dump_c(const char *k, const double2 *v, size_t n) { printf("%s %zu\n", k, n); for (size_t i = 0; i < n; i++) printf("%.17g %.17g\n", v[i].x, v[i].y); }

#define DI(s, f) dump_i(#f, (long long)(s).f)
#define DD(s, f) dump_d(#f, (s).f)

// continuous batch: window / pre-filter tables are null where the mode has none
static void dump_batch(const jb::DemodParams &p, const jb::CfePlan &c, double st_freq, const double2 *cfe_tw, const double *window,
                       const double2 *pre_H, const double2 *pre_tw)
{
    DI(p, kind); DI(p, n_channels); DI(p, cpad); DD(p, Fs); DD(p, fb); DD(p, lockingbw); DD(p, signalthreshold); DD(p, ee);
    DI(p, afc); DI(p, sql); DI(p, cpu_reduce); DI(p, report_ebno); DI(p, ntaps); DI(p, agc_len); DI(p, ebno_len); DI(p, bbnfft);
    DI(p, marg_len); DI(p, dt_len); DI(p, mse_len); DI(p, sps); DD(p, correctionfactor);
    DD(p, res_a1); DD(p, res_a2); DD(p, res_b0); DD(p, res_b1); DD(p, res_b2);
    DD(p, lf_a1); DD(p, lf_a2); DD(p, lf_b0); DD(p, lf_b1); DD(p, lf_b2);
    dump_v("w41v", p.w41v, 4); dump_v("w8v", p.w8v, 4); DI(p, k41); DI(p, k8); DI(p, soft_cap);
    dump_v("taps", p.taps, p.ntaps);
    dump_d("st_freq", st_freq);
    DI(c, nfft); DI(c, n1); DI(c, n2); DI(c, startbin); DI(c, stopbin); DI(c, expectedpeakbin); DI(c, lo); DI(c, hi); DI(c, is8400);
    DD(c, hzperbin);
    dump_c("cfe_tw", cfe_tw, c.nfft);
    if (window) dump_v("cfe_window", window, c.nfft);
    if (pre_H) { dump_c("pre_H", pre_H, 4096); dump_c("pre_tw", pre_tw, 4096); }
}

static void dump_burst(const jb::BurstParams &p, const jb::HilbertStream &h, double freq_center, const double *w_btd1, const double *w_btdiff,
                       const double *w_a1, const double2 *hil_H, const double2 *hil_tw, const double2 *tw32k)
{
    DI(p, kind); DI(p, n_channels); DI(p, cpad); DI(p, sps); DI(p, ntaps); DD(p, spsd); DI(p, tri_nb); DI(p, tri_nt); DI(p, sql);
    dump_v("w41v", p.w41v, 4); dump_v("w8v", p.w8v, 4); DI(p, k41); DI(p, k8);
    DD(p, Fs); DD(p, fb); DD(p, lockingbw); DD(p, signalthreshold); DD(p, ee); DI(p, afc);
    DI(p, agc_len); DI(p, d1_len); DI(p, d2_len); DI(p, btd1_len); DI(p, btma_len); DI(p, mav1_len); DI(p, btdiff_len); DI(p, pd_len); DI(p, tri_sz);
    DI(p, size_base); DI(p, size_top); DI(p, start_processing); DI(p, end_rotation); DI(p, startstopstart);
    DI(p, eb_len); DI(p, agc2_len); DI(p, ds_len); DI(p, d8_k); DI(p, a1_k); DI(p, msema_len); DI(p, soft_cap);
    DD(p, d8_w); DD(p, a1_w); DD(p, btd1_w); DD(p, btdiff_w); DD(p, pd_threshold);
    DD(p, res_a1); DD(p, res_a2); DD(p, res_b0); DD(p, res_b1); DD(p, res_b2); DI(p, astride);
    dump_v("taps", p.taps, p.ntaps);
    dump_d("freq_center", freq_center);
    dump_v("w_btd1", w_btd1, (size_t)p.btd1_len);
    dump_v("w_btdiff", w_btdiff, (size_t)p.btdiff_len);
    dump_v("w_a1", w_a1, (size_t)p.a1_k + 1);
    DI(h, K); DI(h, nfft); DI(h, L);
    dump_c("hil_H", hil_H, h.nfft); dump_c("hil_tw", hil_tw, h.nfft); dump_c("tw32k", tw32k, jb::TRI_N);
}

static void dump_pchannel(const jb::PChanParams &pp)
{
    DI(pp, n_channels); DI(pp, oqpsk); DI(pp, cols); DI(pp, block_len); DI(pp, number_of_bits); DI(pp, bits_in_header);
    DI(pp, total_number_of_bits); DI(pp, paddinglength); DI(pp, dl2_len); DI(pp, info_cap); DI(pp, su_cap); DI(pp, queue);
}

static void dump_rt(const jb::RtParams &rp)
{
    DI(rp, n_channels); DI(rp, oqpsk); DI(rp, ifb); DI(rp, number_of_bits); DI(rp, total_number_of_bits);
}
