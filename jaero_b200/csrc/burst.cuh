// Burst MSK demodulator (K3 acquisition + K4 tail) — device data layout and launch prototypes.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace jb {

static const int BURST_MAXEV = 8;          // trident-buffer fills that may complete within one internal chunk
static const int BURST_CHUNK = 16384;      // internal chunk length (samples); fills complete >= 2*pdet.length apart
static const int TRI_N = 32768;            // FFTr size (burstmskdemodulator.cpp:217)

struct HilbertStream {                     // QJHilbertFilter (DSP.cpp:754-794) as a streaming FFT convolution
    int K, nfft, L;                        // 2048 taps, nfft 8192 -> L = nfft-K+1 = 6145
    double2 *H, *tw;                       // FFT of the zero-padded kernel, W_nfft^k
    double2 *hist, *inblk, *outblk;        // [ch][K-1], [ch][L], [ch][L]
};

// per-channel scalar state of the burst demodulator: doubles BD[idx][cpad], ints BI[idx][cpad]
enum BDIdx {
    BD_AGC_SUM, BD_AGC_VAL, BD_BTMA_SUM_RE, BD_BTMA_SUM_IM, BD_MAV1_SUM, BD_PD_LASTDY, BD_PD_MAXVAL,
    BD_M2_PTR, BD_M2_STEP, BD_M2_FREQ, BD_M2_LAST, BD_MC_PTR, BD_MC_STEP, BD_MC_FREQ, BD_MC_LAST,
    BD_ST_PTR, BD_ST_STEP, BD_ST_FREQ, BD_ST_LAST, BD_SH_PTR, BD_SH_STEP, BD_SH_FREQ, BD_SH_LAST,
    BD_VOL_GAIN, BD_MSE, BD_MSEMA_SUM, BD_ROT_RE, BD_ROT_IM, BD_ROT_FREQ, BD_STR_RE, BD_STR_IM, BD_SAV_RE, BD_SAV_IM,
    BD_EB_SUM1, BD_EB_SUM2, BD_EB_EBNO, BD_AGC2_SUM, BD_AGC2_VAL, BD_RES_X1, BD_RES_X2, BD_RES_Y1, BD_RES_Y2, BD_DIFF_LAST,
    BD_LAST_EBNO_EMIT,
    // burst OQPSK only
    BD_SR_PTR, BD_SR_STEP, BD_SR_FREQ, BD_SR_LAST,           // st_osc_ref (BD_SH_* holds st_osc_quarter)
    BD_DLY_S0, BD_DLY41_0, BD_DLY41_1, BD_DLY41_2, BD_DLY42_0, BD_DLY42_1, BD_DLY42_2, BD_DLY8_0, BD_DLY8_1, BD_DLY8_2,
    BD_SIG2L_RE, BD_SIG2L_IM, BD_PTD_RE, BD_PTD_IM, BD_LASTMSE,
    BD_COUNT
};
enum BIIdx {
    BI_PD_CNTDOWN, BI_PD_MAXPOSCNT, BI_TRI_PTR, BI_TRI_SLOT, BI_NEV, BI_CNTR, BI_STARTSTOP, BI_DCD,
    BI_FIR_POS, BI_A1_POS, BI_EB_POS, BI_AGC2_POS, BI_DS_POS, BI_D8_POS, BI_MSEMA_POS,
    BI_SOFT_COUNT, BI_SOFT_PENDING, BI_SOFT_OVERFLOW, BI_SIG_TRUE, BI_SIG_FALSE, BI_EBNO_EMITS,
    BI_YUI, BI_INSERTPREAMBLE,
    BI_COUNT
};

struct BurstParams {
    int kind;                              // 0 = burst MSK, 1 = burst OQPSK
    int n_channels, cpad, sps, ntaps;
    double spsd;                           // SamplesPerSymbol as the reference holds it (9.142857... for OQPSK)
    int tri_nb, tri_nt;                    // samples of the base / top trident sections
    int sql;
    double w41v[4], w8v[4]; int k41, k8;   // OQPSK timing delays (T/4, T/8): weight per ring position
    const double *btd1_wv, *btdiff_wv, *a1_wv;   // Delay<> interpolation weight per ring position
    double Fs, fb, lockingbw, signalthreshold, ee;
    int afc;
    int agc_len, d1_len, d2_len, btd1_len, btma_len, mav1_len, btdiff_len, pd_len, tri_sz;      // ring sizes (entries)
    int size_base, size_top, start_processing, end_rotation, startstopstart;
    int eb_len, agc2_len, ds_len, d8_k, a1_k, msema_len, soft_cap;
    double d8_w, a1_w, btd1_w, btdiff_w, pd_threshold;
    double res_a1, res_a2, res_b0, res_b1, res_b2;
    double *BD; int *BI;
    // lock-step rings [slot][cpad]
    double *agc_ring, *d2_ring, *mav1_ring, *btdiff_ring, *pd1_ring, *pd2_ring, *pd3_ring;
    double2 *d1_ring, *btd1_ring, *btma_ring;
    // per-channel-position rings [slot][cpad]
    double *a1_ring, *eb1_ring, *eb2_ring, *agc2_ring, *d8_ring, *msema_ring, *fir_re, *fir_im;
    double2 *ds_ring;
    double *tri;                           // [ch][BURST_MAXEV][tri_sz] trident buffers (one slot per fill)
    int *ev_sample;                        // [ch][BURST_MAXEV] chunk-relative sample index at which a fill completed
    double *ev_result;                     // [ch][BURST_MAXEV][8]: minvalbin, minval, maxtoppos, maxtopposhigh, arg(out_base[minvalbin])
    double2 *analytic;                     // [ch][astride] Hilbert output of the current chunk
    double *vtd;                           // [ch][astride] val_to_demod of the current chunk
    size_t astride;
    int16_t *soft;                         // [ch][soft_cap]
    const double *sin_t, *cos_t;
    double taps[160];                      // matched-filter taps of THIS demodulator (kernel parameter block; MAX_TAPS of demod.cuh)
};

int hilbert_exchange_launch(const HilbertStream &h, const BurstParams &p, const int16_t *pcm, size_t stride, int pcm0, int i0, int i1, int fill0, cudaStream_t s);
int hilbert_block_launch(const HilbertStream &h, int n_channels, int first_block, cudaStream_t s);
int burst_front_launch(const BurstParams &p, long long sample0, int n, cudaStream_t s);
int burst_trident_launch(const BurstParams &p, double2 *work_a, double2 *work_b, const double2 *tw16k, double *absbuf, cudaStream_t s, long long *launches);
int burst_back_launch(const BurstParams &p, long long sample0, int n, int new_write, cudaStream_t s);
int burst_trident_fft_launch(const BurstParams &p, const int *d_ev_list, int n_events, double2 *wa, double2 *wb, const double2 *tw, cudaStream_t s);

} // namespace jb
