// K1a (10500 bps) — warp-specialised OQPSK demodulator segment kernel.
//
// Same arithmetic, statement for statement, as oqpsk_segment_kernel<false> (oqpsk_demod.cu), i.e. as
// OqpskDemodulator::writeData (JAERO/oqpskdemodulator.cpp:334-627). What changes is who executes it: the per-sample
// recursion of one channel is a feedback loop (carrier NCO -> FIR -> AGC -> timing -> strobe -> carrier NCO), so a
// single thread per channel is bound by the length of its dependent instruction chain (~1500 instructions per sample),
// not by HBM. The chain is cut where the reference's own structure allows it:
//
//   * the FIR output of sample n excludes the sample written at n (DSP.cpp:292-304), so everything from the FIR to the
//     timing-error detector's input (FIR, EbNo, AGC, clip, T/4 delays, resonator, T/8 delay) is FEED-FORWARD from the
//     mixed samples up to n-1;
//   * the symbol-rate tail after the carrier update (bias rotate, 400-symbol delay, MSE, soft bits) feeds nothing back
//     inside a call.
//
// Six warps of one CTA each own a slice of the per-sample work of the same 32 channels (lane = channel in every warp)
// and hand their results to the next warp through shared memory, ordered by named barriers (bar.arrive / bar.sync on
// alternating ids, one producer warp + one consumer warp per barrier):
//
//   warp F  input: PCM tiles (TMA), coarse-estimator ring write (mixer_center); 55-tap FIR of the mixed samples -> dval, sig2raw
//   warp E  EbNo + AGC running sums (TMA-staged ring tiles), AGC gain, clip, timing feed-forward chain     -> sig2, st_eta, d8out
//   warp T  symbol-timing PLL: arg of the timing-error phasor, st_osc nudges, strobe test                  -> (strobe, fraction)
//   warp K1 strobe interpolation, carrier error (tanh x2), loop filter                                      -> ct_ec, (pt_qpsk, ct_ec)
//   warp K2 carrier NCO (phase / frequency update, advance, table look-up); mixes the NEXT input sample
//           and puts it into the FIR window                                                                 -> cval
//   warp S  marg MA(800), 400-symbol delay, bias rotate, MSE, soft bits
//
// The only loop that remains serial is K2(n-1) -> newest FIR tap -> E(n+1) -> T(n+1) -> K1(n+1) -> K2(n+1): it advances two
// samples per turn; K1(n+1) overlaps K2(n). F, S and the bulk of the FIR are off that loop entirely. Back-pressure from S
// (slot free) uses two mbarriers: the 16 named barriers are all taken by the seven forward signals.
#include "demod_device.cuh"

namespace jb {

static const int PP_THREADS = 224;                  // seven role warps
// shared memory map (bytes): FIR windows | ring tiles x6 | PCM tiles x2 | mbarriers | hand-off slots
static const int PP_HF = 16;                        // doubles per lane in a hand-off slot
static const int PP_SM_HAND = 2 * PP_HF * 32 * 8;  // [2 slots][PP_HF doubles][32 lanes]
static const int PP_NBUF = 3;                       // ring-tile buffers: a tile is reloaded into the buffer stored a whole tile earlier,
                                                    // so the writer never waits for a bulk store to drain (with 2 buffers it stalled
                                                    // ~12 000 cycles at every 32-sample tile boundary: 19 % of the launch)
static const int PP_SM_BASE = OQ_SM_FIR + 3 * PP_NBUF * OQ_SM_RING + 128;           // FIR windows | ring tiles | 16 mbarriers
static const int PP_DV = 64;                        // input-sample ring (doubles per lane): two tiles of 32, warp A -> warp K2
static const int PP_SM_DV = PP_DV * 32 * 8;
static const int PP_SM_BBST = 8 * 32 * 16;          // one 128-byte estimator-ring line per lane, staged before it is written
static const int PP_SM_TOTAL = PP_SM_BASE + PP_SM_HAND + PP_SM_DV + PP_SM_BBST;
// named barriers (0 is __syncthreads)
enum { BAR_X = 1, BAR_YT = 3, BAR_Z = 5, BAR_W = 7, BAR_P = 9, BAR_YK = 11, BAR_U = 13 };

// Producer side of a hand-off: st.shared, membar.cta, bar.arrive; consumer side bar.sync, ld.shared. (Without the membar the
// kernel is 1.2 % faster and every parity test still passes - bar.arrive is not documented to order the producer's stores, so it stays.)
#define PP_HANDOFF_FENCE() __threadfence_block()
__device__ __forceinline__ void nb_arrive(int id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void nb_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

#define LD(idx) p.D[(size_t)(idx) * cpad + ch]
#define LI(idx) p.I[(size_t)(idx) * cpad + ch]

#define TR(k) do { if (a.trace && blockIdx.x == 0 && lane == 0 && j >= a.trace_j0 && j < a.trace_j0 + 64) a.trace[(j - a.trace_j0) * 16 + (k)] = clock64(); } while (0)
#define PP_WAIT(idx) do { mbar_wait(&bars[(idx)], (phases >> (idx)) & 1u); phases ^= (1u << (idx)); } while (0)
__global__ void __launch_bounds__(PP_THREADS)
oqpsk_pipe_kernel(const __grid_constant__ DemodParams p, const SegmentArgs a, const int16_t *__restrict__ pcm, size_t stride)
{
    extern __shared__ __align__(128) unsigned char pp_smem_raw[];
    double *s_re = reinterpret_cast<double *>(pp_smem_raw);   // [OQ_FIRROWS][32]
    double *s_im = s_re + OQ_FIRROWS * OQ_THREADS;
    double *t_agc = reinterpret_cast<double *>(pp_smem_raw + OQ_SM_FIR);          // [PP_NBUF][T][32]
    double *t_e1 = t_agc + PP_NBUF * OQ_T * OQ_THREADS;
    double *t_e2 = t_e1 + PP_NBUF * OQ_T * OQ_THREADS;
    // mbarriers: 0-2 ring tiles, 3-4 input tile full (A -> K2), 5-6 symbol slot free (S -> K1), 7-8 input tile empty (K2 -> A)
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(pp_smem_raw + OQ_SM_FIR + 3 * PP_NBUF * OQ_SM_RING);
    double *hand = reinterpret_cast<double *>(pp_smem_raw + PP_SM_BASE);           // [2][PP_HF][32]
    double *dv = reinterpret_cast<double *>(pp_smem_raw + PP_SM_BASE + PP_SM_HAND);               // [PP_DV][32]
    double2 *bbst = reinterpret_cast<double2 *>(pp_smem_raw + PP_SM_BASE + PP_SM_HAND + PP_SM_DV); // [8][32]
    // Role ids: F 0, E 1, T 2, K1 3, K2 4, S 5, A 6 = physical warp. (Warps w and w+4 share an SM sub-partition and its FP64
    // pipe. Other placements were measured on B200 inside one GPU call, 9-warp CTAs with placeholder warps: {F,S,A | E | T | K1,K2},
    // {F,A | E,S | T | K1,K2}, {F,S | E,A | T | K1,K2}: all 8 % slower per epoch than this one.)
    const int lane = threadIdx.x & 31;
    const int warp = (int)(threadIdx.x >> 5);
    // Which channel this lane carries. Channels are independent, so the library may seat them as it likes: it regroups them by
    // symbol-timing phase (capi_batch.cu, regroup) so that the 32 channels of a CTA strobe on the same samples - the expensive
    // carrier-update path of warps K1 / K2 then runs on one sample in nine instead of (some lane) on every sample. All state
    // stays indexed by channel; only the sample-rate rings, which are laid out by seat, move when the seating changes.
    const int seat = blockIdx.x * OQ_THREADS + lane;
    const int ch = p.chan_of ? p.chan_of[seat] : seat;       // dead lanes run on their (allocated) pad column with zero input
    const bool live = ch < p.n_channels;
    const size_t cpad = p.cpad;
    if (threadIdx.x == 0) { for (int k = 0; k < 3; k++) mbar_init(&bars[k], 1); for (int k = 3; k < 9; k++) mbar_init(&bars[k], 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();                                           // (0) mbarriers usable

    const int nB = (a.i1 - a.i0) - (a.stop_after_a ? 1 : 0);             // samples whose loop body runs in this launch
    const long long S0 = a.sample0;
    const double Fs = p.Fs;
    const double *__restrict__ cos_t = p.cos_t, *__restrict__ sin_t = p.sin_t;
    // hand-off slot layout: slot s, field f -> hand[(s * 12 + f) * 32 + lane]
    //   f 0,1: sig2raw (F->E)   f 2,3: sig2 (E->K)   f 4,5: st_eta, d8out (E->T)   f 6..9: pt_qpsk.x, pt_qpsk.y, ct_ec, flag (K->S)
    //   f 10,11: strobe flag, FractionOfSampleItPassesBy (T->K1)   f 12: next input sample (F->K2)   f 13 (slot 0): first input sample (F->K2)
    //   f 14,15: carrier-update flag, ct_ec (K1->K2)
#define HAND(s, f) hand[((s) * PP_HF + (f)) * 32 + lane]

    // ======================================================================================= warp K2: carrier NCO + mixer
    if (warp == 4) {
        Osc m2 = {LD(D_M2_PTR), LD(D_M2_STEP), LD(D_M2_FREQ), LD(D_M2_LAST)};
        // ---- FreqOffsetEstimateSlot (oqpskdemodulator.cpp:629-677), re-entrant in the reference: it runs after the ring
        // write and before the mixer of the same sample.
        if (a.apply_cfe) {
            Osc mc = {LD(D_MC_PTR), LD(D_MC_STEP), LD(D_MC_FREQ), LD(D_MC_LAST)};
            const double mse = LD(D_MSE);
            const int dcd = LI(I_DCD);
            int countdown = LI(I_COUNTDOWN), countdown2 = LI(I_COUNTDOWN2);
            double est = 0.0;
            if (a.cfe_wait > 0) {
                // The estimator of this trigger runs concurrently (capi_batch.cu). Its result only enters the arithmetic below when
                // the channel is unlocked / has no carrier detect, and its state (y[], emptyingcountdown) is only touched by
                // the AFC re-centre: channels in neither case proceed without it.
                const bool recentre = (p.afc) && (mse < p.signalthreshold) && (fabs(m2.freq - mc.freq) > 3.0) && (countdown <= 0);
                const bool need = (mse > p.signalthreshold) || (!dcd) || recentre;
                if (__any_sync(0xffffffffu, need)) {
                    const volatile int *flag = p.cfe_flag;
                    while (*flag < a.cfe_wait) __nanosleep(256);
                    __threadfence();
                }
                if (need) est = __ldcg(p.cfe_est_out + ch);
            } else est = p.cfe_est_out[ch];
            if ((mse < p.signalthreshold) && (!dcd)) {                        // :642-650
                if (countdown2 > 0) countdown2--;
                else osc_set_freq(m2, mc.freq + est, p.Fs);
            } else countdown2 = 5;
            if ((mse > p.signalthreshold) && (fabs(m2.freq - (mc.freq + est)) > 3.0))    // :653-657
                osc_set_freq(m2, mc.freq + est, p.Fs);
            if ((p.afc) && (mse < p.signalthreshold) && (fabs(m2.freq - mc.freq) > 3.0)) {   // :658-669
                if (countdown > 0) countdown--;
                else {
                    osc_set_freq(mc, m2.freq, p.Fs);
                    if (mc.freq < p.lockingbw / 2.0) osc_set_freq(mc, p.lockingbw / 2.0, p.Fs);
                    if (mc.freq > (p.Fs / 2.0 - p.lockingbw / 2.0)) osc_set_freq(mc, p.Fs / 2.0 - p.lockingbw / 2.0, p.Fs);
                    LI(I_EMPTYING) = 4;                                       // CoarseFreqEstimate::bigchange (coarsefreqestimate.cpp:84-88)
                    LI(I_ZERO_BB) = 1;                                        // y[]=20 is applied by the estimator kernel on its next run
                    double2 *rowz = p.bb + (size_t)ch * p.bb_len;             // :667 bbcycbuff[j]=0
                    if (live) for (int j = 0; j < p.bb_len; j++) rowz[j] = make_double2(0.0, 0.0);
                    LD(D_MC_STEP) = mc.step; LD(D_MC_FREQ) = mc.freq;         // warp F reloads mixer_center after the barrier
                }
            } else countdown = 4;
            if (mse > p.signalthreshold) { LI(I_SIG_FALSE) = LI(I_SIG_FALSE) + 1; if (p.wire_sigstat) { const int ln_ = LI(I_LOST_N); if (ln_ < LOST_CAP) p.lost_pos[(size_t)ln_ * cpad + ch] = LI(I_SOFT_COUNT); LI(I_LOST_N) = ln_ + 1; LI(I_DCD) = 0; } }   // :674-675
            else LI(I_SIG_TRUE) = LI(I_SIG_TRUE) + 1;
            LI(I_COUNTDOWN) = countdown; LI(I_COUNTDOWN2) = countdown2;
        }
        __syncthreads();                                       // (1) slot done, FIR window resident
        if (nB > 0) {
            double c2_re, c2_im;
            { const int t = osc_index(m2.ptr); c2_re = cos_t[t]; c2_im = sin_t[t]; }
            int fir_pos = (int)(S0 % OQ_NT1);                  // slot of the sample being mixed
            unsigned kph = 0u;                                 // parities of the two input-tile-full mbarriers
            mbar_wait(&bars[3], 0u); kph ^= 1u;                // input tile 0 (warp A)
            {   // cval of the first sample (:453)
                const double dval = dv[lane];
                const double cre = c2_re * dval, cim = c2_im * dval;
                s_re[fir_pos * OQ_THREADS + lane] = cre; s_re[(fir_pos + OQ_NT1) * OQ_THREADS + lane] = cre;
                s_im[fir_pos * OQ_THREADS + lane] = cim; s_im[(fir_pos + OQ_NT1) * OQ_THREADS + lane] = cim;
                fir_pos++; if (fir_pos >= OQ_NT1) fir_pos = 0;
                PP_HANDOFF_FENCE();
                nb_arrive(BAR_X + 0);                          // X_0
            }
            for (int j = 0; j < nB; j++) {
                const int sl = j & 1;
                // speculative request for mixer2's next entry (right unless this sample turns out to be a carrier-update strobe)
                const int m2_spec = osc_next_index(m2);
                const double n2_re = __ldcg(cos_t + m2_spec), n2_im = __ldcg(sin_t + m2_spec);
                double dnext = 0.0;                            // input sample j+1, decoded by warp A a tile or two ahead
                if (j + 1 < nB) {
                    const int e = j + 1, tb = (e >> 5) & 1;
                    if ((e & 31) == 0) { mbar_wait(&bars[3 + tb], (kph >> tb) & 1u); kph ^= (1u << tb); }
                    dnext = dv[(e & (PP_DV - 1)) * 32 + lane];
                    if ((e & 31) == 31) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bars[7 + tb])) : "memory");   // tile read
                }
                // a carrier update moves the pointer by ct_ec degrees = 55.6 * ct_ec entries: a few entries in lock, so the
                // entry needed after an update sits in the speculated 128-byte line or one of its neighbours
                nb_sync(BAR_P + sl);                           // P_j: carrier error of this sample (warp K1)
                TR(8);
                const double upd = HAND(sl, 14), ct_ec = HAND(sl, 15);
                if (upd != 0.0) {                                                 // :518-525, fb > 8400 (the host only uses this kernel there)
                    osc_increase_phase_deg(m2, 1.0 * ct_ec);
                    osc_set_freq(m2, (0.01 * ct_ec) + m2.freq, Fs);
                }
                osc_next_frame(m2);                                               // :600 (st_osc / st_osc_ref live in warp T, mixer_center in warp T)
                {
                    const int t = osc_index(m2.ptr);
                    if (t == m2_spec) { c2_re = n2_re; c2_im = n2_im; } else { c2_re = __ldcg(cos_t + t); c2_im = __ldcg(sin_t + t); }
                }
                TR(13);
                if (j + 1 < nB) {   // the next sample's mixed value enters the FIR ring (:453-456)
                    const double cre = c2_re * dnext, cim = c2_im * dnext;
                    s_re[fir_pos * OQ_THREADS + lane] = cre; s_re[(fir_pos + OQ_NT1) * OQ_THREADS + lane] = cre;
                    s_im[fir_pos * OQ_THREADS + lane] = cim; s_im[(fir_pos + OQ_NT1) * OQ_THREADS + lane] = cim;
                    fir_pos++; if (fir_pos >= OQ_NT1) fir_pos = 0;
                    PP_HANDOFF_FENCE();
                    nb_arrive(BAR_X + ((j + 1) & 1));          // X_{j+1}
                    TR(9);
                }
            }
        }
        LD(D_M2_PTR) = m2.ptr; LD(D_M2_STEP) = m2.step; LD(D_M2_FREQ) = m2.freq; LD(D_M2_LAST) = m2.last;
    }
    // ======================================================================================= warp K1: carrier error
    else if (warp == 3) {
        Biquad lf = {LD(D_LF_X1), LD(D_LF_X2), LD(D_LF_Y1), LD(D_LF_Y2)};
        double2 sig2_last = make_double2(LD(D_SIG2L_RE), LD(D_SIG2L_IM));
        double2 pt_d = make_double2(LD(D_PTD_RE), LD(D_PTD_IM));
        int yui = LI(I_YUI), sig2l_init = LI(I_SIG2L_INIT);
        // tanh(pt_d.x) only changes when pt_d does (on the strobes of the other arm): it is evaluated right after that strobe's
        // hand-off instead of on the carrier-update sample, where it sat on the feedback loop
        double th_ptd = tanh(pt_d.x);
        bool th_stale = false;
        __syncthreads();                                       // (1)
        {
            unsigned vph = 0u;                                 // parities of the two slot-free mbarriers
            for (int j = 0; j < nB; j++) {
                const int sl = j & 1;
                nb_sync(BAR_YK + sl);                          // sig2 of this sample (warp E)
                double2 sig2 = make_double2(HAND(sl, 2), HAND(sl, 3));
                nb_sync(BAR_U + sl);                           // strobe decision of this sample (warp T)
                const double strobe = HAND(sl, 10), frac = HAND(sl, 11);
                TR(6);
                if (!sig2l_init) { sig2_last = sig2; sig2l_init = 1; }            // :487 static initialiser
                double sy_flag = 0.0, sy_x = 0.0, sy_y = 0.0, sy_ec = 0.0, k2_upd = 0.0, k2_ec = 0.0;
                if (strobe != 0.0) {                                              // :488
                    const double pt_last = frac, pt_this = 1.0 - pt_last;
                    const double2 pt = make_double2(pt_this * sig2.x + pt_last * sig2_last.x, pt_this * sig2.y + pt_last * sig2_last.y);
                    yui ^= 1;                                                     // yui++; yui%=2;
                    if (!yui) { pt_d = pt; th_stale = true; }
                    else {
                        const double2 pt_qpsk = make_double2(pt.x, pt_d.y);       // :503
                        const double ct_xt = tanh(pt.y) * pt.x;
                        const double ct_xt_d = th_ptd * pt_d.y;
                        double ct_ec = ct_xt_d - ct_xt;
                        if (ct_ec > M_PI) ct_ec = M_PI;
                        if (ct_ec < -M_PI) ct_ec = -M_PI;
                        // :518-525 (fb > 8400: the loop filter sits in front of the NCO update; the host only uses this kernel there)
                        ct_ec = biquad_update(lf, ct_ec, p.lf_a1, p.lf_a2, p.lf_b0, p.lf_b1, p.lf_b2);
                        if (ct_ec > M_PI_2) ct_ec = M_PI_2;
                        if (ct_ec < -M_PI_2) ct_ec = -M_PI_2;
                        k2_upd = 1.0; k2_ec = ct_ec;
                        sy_flag = 1.0; sy_x = pt_qpsk.x; sy_y = pt_qpsk.y; sy_ec = ct_ec;
                    }
                }
                sig2_last = sig2;                                                 // :596
                // slot sl's K1->K2 fields were read by K2(j-2), which precedes X_{j-1} -> ... -> U_j: free
                HAND(sl, 14) = k2_upd; HAND(sl, 15) = k2_ec;
                PP_HANDOFF_FENCE();
                nb_arrive(BAR_P + sl);                         // P_j
                TR(7);
                // symbol hand-off to warp S; slot reuse is gated by S's arrival on the slot's mbarrier
                if (j >= 2) { mbar_wait(&bars[5 + sl], (vph >> sl) & 1u); vph ^= (1u << sl); }
                HAND(sl, 6) = sy_x; HAND(sl, 7) = sy_y; HAND(sl, 8) = sy_ec; HAND(sl, 9) = sy_flag;
                PP_HANDOFF_FENCE();
                nb_arrive(BAR_W + sl);                         // W_j
                if (th_stale) { th_ptd = tanh(pt_d.x); th_stale = false; }
            }
        }
        LD(D_LF_X1) = lf.x1; LD(D_LF_X2) = lf.x2; LD(D_LF_Y1) = lf.y1; LD(D_LF_Y2) = lf.y2;
        LD(D_SIG2L_RE) = sig2_last.x; LD(D_SIG2L_IM) = sig2_last.y;
        LD(D_PTD_RE) = pt_d.x; LD(D_PTD_IM) = pt_d.y;
        LI(I_YUI) = yui; LI(I_SIG2L_INIT) = sig2l_init;
    }
    // ======================================================================================= warp S: symbol-rate tail
    else if (warp == 5) {
        double marg_sum = LD(D_MARG_SUM), marg_val = LD(D_MARG_VAL);
        double pm_sum = LD(D_MSE_PM_SUM), ma_sum = LD(D_MSE_MA_SUM), mse = LD(D_MSE);
        double lastmse = LD(D_LASTMSE);
        double2 sc0 = make_double2(LD(D_SCAT0_RE), LD(D_SCAT0_IM)), sc1 = make_double2(LD(D_SCAT1_RE), LD(D_SCAT1_IM));
        int marg_pos = LI(I_MARG_POS), dt_pos = LI(I_DT_POS), mse_pos = LI(I_MSE_POS);
        int soft_count = LI(I_SOFT_COUNT), soft_pending = LI(I_SOFT_PENDING), soft_overflow = LI(I_SOFT_OVERFLOW);
        if (a.new_write) lastmse = mse;                                       // oqpskdemodulator.cpp:339
        const int marg_len = p.marg_len, dt_len = p.dt_len, mse_len = p.mse_len;
        const double thr = p.signalthreshold;
        const double r_marg = 1.0 / ((double)marg_len), r_mse = 1.0 / ((double)mse_len);
        double sy_marg_old = p.marg_ring[(size_t)marg_pos * cpad + ch];
        double sy_pm_old = p.mse_pm[(size_t)mse_pos * cpad + ch];
        double sy_ma_old = p.mse_ma[(size_t)mse_pos * cpad + ch];
        double2 sy_dt_old;
        { int r = dt_pos + 1; if (r >= dt_len) r = 0; sy_dt_old = p.dt_ring[(size_t)r * cpad + ch]; }
        __syncthreads();                                       // (1)
        for (int j = 0; j < nB; j++) {
            const int sl = j & 1;
            nb_sync(BAR_W + sl);                               // W_j
            const double fx = HAND(sl, 6), fy = HAND(sl, 7), fec = HAND(sl, 8), fl = HAND(sl, 9);
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bars[5 + sl])) : "memory");   // slot read (release)
            if (fl != 0.0) {
                double2 pt_qpsk = make_double2(fx, fy);
                const double ct_ec = fec;
                {   // marg->UpdateSigned(ct_ec)  MA(800)  (:535, DSP.cpp:418-426)
                    marg_sum = marg_sum - sy_marg_old;
                    marg_sum = marg_sum + (ct_ec);
                    p.marg_ring[(size_t)marg_pos * cpad + ch] = (ct_ec);
                    marg_pos++; if (marg_pos >= marg_len) marg_pos = 0;
                    marg_val = div_exact(marg_sum, (double)marg_len, r_marg);
                }
                {   // dt.update(pt_qpsk): 400-symbol delay (:536, DSP.h:455-460)
                    p.dt_ring[(size_t)dt_pos * cpad + ch] = pt_qpsk;
                    dt_pos++; if (dt_pos >= dt_len) dt_pos = 0;
                    pt_qpsk = sy_dt_old;                                  // requested after the previous strobe
                }
                pt_qpsk = cmul(pt_qpsk, make_double2(cos(marg_val), sin(marg_val)));   // :537
                sc1 = sc0; sc0 = pt_qpsk;                                              // pointbuff (:546), decimated
                {   // MSEcalc::Update (DSP.cpp:451-463)
                    const size_t e = (size_t)mse_pos * cpad + ch;
                    const double ab = hypot(pt_qpsk.x, pt_qpsk.y);
                    pm_sum = pm_sum - sy_pm_old; pm_sum = pm_sum + fabs(ab); p.mse_pm[e] = fabs(ab);
                    double mu = div_exact(pm_sum, (double)mse_len, r_mse);
                    if (mu < 0.000001) mu = 0.000001;
                    const double r2 = sqrt(2.0);
                    const double tre = (r2 * pt_qpsk.x) / mu, tim = (r2 * pt_qpsk.y) / mu;
                    const double tda = (fabs(tre) - 1.0), tdb = (fabs(tim) - 1.0);
                    const double v = (tda * tda) + (tdb * tdb);
                    ma_sum = ma_sum - sy_ma_old; ma_sum = ma_sum + fabs(v); p.mse_ma[e] = fabs(v);
                    mse_pos++; if (mse_pos >= mse_len) mse_pos = 0;
                    mse = div_exact(ma_sum, (double)mse_len, r_mse);
                }
                // operands of the next strobe pair (slots written >= 400 symbols ago)
                sy_marg_old = p.marg_ring[(size_t)marg_pos * cpad + ch];
                sy_pm_old = p.mse_pm[(size_t)mse_pos * cpad + ch];
                sy_ma_old = p.mse_ma[(size_t)mse_pos * cpad + ch];
                { int r = dt_pos + 1; if (r >= dt_len) r = 0; sy_dt_old = p.dt_ring[(size_t)r * cpad + ch]; }
                if (live && mse < thr) {                                  // :565
                    push_soft(p, ch, soft_count, soft_pending, soft_overflow, q_round(0.75 * pt_qpsk.y * 127.0 + 128.0));
                    push_soft(p, ch, soft_count, soft_pending, soft_overflow, q_round(0.75 * pt_qpsk.x * 127.0 + 128.0));
                    if (soft_pending >= 32) {                             // :583-592
                        if (!p.sql || mse < thr || lastmse < thr) soft_count += soft_pending;
                        soft_pending = 0;
                    }
                }
            }
        }
        LD(D_MARG_SUM) = marg_sum; LD(D_MARG_VAL) = marg_val;
        LD(D_MSE_PM_SUM) = pm_sum; LD(D_MSE_MA_SUM) = ma_sum; LD(D_MSE) = mse;
        LD(D_LASTMSE) = lastmse;
        LD(D_SCAT0_RE) = sc0.x; LD(D_SCAT0_IM) = sc0.y; LD(D_SCAT1_RE) = sc1.x; LD(D_SCAT1_IM) = sc1.y;
        LI(I_MARG_POS) = marg_pos; LI(I_DT_POS) = dt_pos; LI(I_MSE_POS) = mse_pos;
        LI(I_SOFT_COUNT) = soft_count; LI(I_SOFT_PENDING) = soft_pending; LI(I_SOFT_OVERFLOW) = soft_overflow;
    }
    // ======================================================================================= warp T: symbol-timing PLL
    else if (warp == 2) {
        Osc st = {LD(D_ST_PTR), LD(D_ST_STEP), LD(D_ST_FREQ), LD(D_ST_LAST)};
        const double sr_freq = LD(D_SR_FREQ);                  // st_osc_ref: only its (constant) frequency is read here; warp A advances it
        __syncthreads();                                       // (1)
        const double ee = p.ee;
        double cs_re, cs_im;
        { const int t = osc_index(st.ptr); cs_re = cos_t[t]; cs_im = sin_t[t]; }
        for (int j = 0; j < nB; j++) {
            const int sl = j & 1;
            // speculative request for st_osc's next table entry, issued before this sample's timing nudges are known (they move
            // the pointer by a fraction of an entry): the L2 round trip of the look-up was the longest item of this warp's
            // serial chain (atan2 -> nudges -> advance -> index -> load -> next sample's phasor)
            const int st_spec = osc_next_index(st);
            const double ns_re = cos_t[st_spec], ns_im = sin_t[st_spec];
            nb_sync(BAR_YT + sl);                              // st_eta, d8out of this sample (warp E)
            const double st_eta = HAND(sl, 4), d8out = HAND(sl, 5);
            TR(4);
            const double2 st_out = cmul(make_double2(cs_re, cs_im), make_double2(st_eta, -d8out));   // :478-479
            const double st_angle_error = atan2_fast(st_out.y, st_out.x);     // :480 std::arg
            TR(11);
            osc_set_freq(st, (-st_angle_error * 0.00000001) + st.freq, Fs);   // :481 IncreseFreqHz
            osc_advance_fraction_of_wave(st, div_exact(-st_angle_error * 0.01, 360.0, 1.0 / 360.0)); // :482
            if (st.freq < (sr_freq - 0.1)) osc_set_freq(st, (sr_freq - 0.1), Fs);
            if (st.freq > (sr_freq + 0.1)) osc_set_freq(st, (sr_freq + 0.1), Fs);
            double frac = 0.0;
            const bool strobe = osc_have_passed_point(st, ee, frac);          // :488
            // slot sl's T->K1 fields were read by K1(j-2), which precedes X_{j-1} -> Z_j -> (E) -> this point: free
            HAND(sl, 10) = strobe ? 1.0 : 0.0; HAND(sl, 11) = frac;
            PP_HANDOFF_FENCE();
            nb_arrive(BAR_U + sl);
            TR(5);
            osc_next_frame(st);                                               // :602 (st_osc_ref, :603, advances in warp A)
            { const int t = osc_index(st.ptr); if (t == st_spec) { cs_re = ns_re; cs_im = ns_im; } else { cs_re = cos_t[t]; cs_im = sin_t[t]; } }
        }
        LD(D_ST_PTR) = st.ptr; LD(D_ST_STEP) = st.step; LD(D_ST_FREQ) = st.freq; LD(D_ST_LAST) = st.last;
    }
    // ======================================================================================= warp E: envelope chain
    else if (warp == 1) {
        double agc_sum = LD(D_AGC_SUM), agc_val = LD(D_AGC_VAL);
        double eb_sum1 = LD(D_EB_SUM1), eb_sum2 = LD(D_EB_SUM2), eb_ebno = LD(D_EB_EBNO);
        double dly_s0 = LD(D_DLY_S0);
        double d41_0 = LD(D_DLY41_0), d41_1 = LD(D_DLY41_1), d41_2 = LD(D_DLY41_2);
        double d42_0 = LD(D_DLY42_0), d42_1 = LD(D_DLY42_1), d42_2 = LD(D_DLY42_2);
        double d8_0 = LD(D_DLY8_0), d8_1 = LD(D_DLY8_1), d8_2 = LD(D_DLY8_2);
        Biquad res = {LD(D_RES_X1), LD(D_RES_X2), LD(D_RES_Y1), LD(D_RES_Y2)};
        const int agc_len = p.agc_len, eb_len = p.ebno_len;
        const bool ebno_on = p.report_ebno != 0;
        const double fbr = p.fb, r_agc = 1.0 / ((double)agc_len);
        const double res_a1 = p.res_a1, res_a2 = p.res_a2, res_b0 = p.res_b0, res_b1 = p.res_b1, res_b2 = p.res_b2;
        long long S = S0;
        int p41 = (int)(S % (p.k41 + 1)), p8 = (int)(S % (p.k8 + 1));   // Delay<> ring positions (lock-step)
        const int k41 = p.k41, k8 = p.k8;
        const long long S_end = S + nB;
        const int eb_from_j = (a.i1 - a.i0) - OQ_EBNO_TAIL;       // same read-out window as oqpsk_segment_kernel
        __syncthreads();                                       // (1)
        if (nB > 0) {
            // Ring layout of THIS kernel (the 10500 bps pipeline owns its batch's rings): [cta][slot][32 lanes], so the 32 slots x 32
            // channels of a tile are one contiguous 8 KB block and move with ONE bulk copy per ring, issued by lane 0. (With the
            // [slot][cpad] layout every lane issued its own 256-byte row copy; UBLKCP is a warp-uniform instruction, so those 96
            // stores + 96 loads per tile boundary were issued one after the other: a 12 000-cycle stall every 32 samples.)
            auto ring_tile = [&](double *ring, int len, long long tile) -> double * {
                return ring + ((size_t)blockIdx.x * len + (size_t)((tile * OQ_T) % len)) * OQ_THREADS;
            };
            const unsigned ring_tx = (ebno_on ? 3u : 1u) * OQ_SM_RING;
            auto ring_load = [&](long long tile) {
                const int b = (int)(tile % PP_NBUF);
                fence_proxy_async();                                  // every lane: its generic accesses to the buffer precede the copy
                __syncwarp();
                if (lane == 0) {
                    mbar_expect_tx(&bars[b], ring_tx);
                    bulk_g2s(t_agc + b * OQ_T * OQ_THREADS, ring_tile(p.agc_ring, agc_len, tile), OQ_SM_RING, &bars[b]);
                    if (ebno_on) {
                        bulk_g2s(t_e1 + b * OQ_T * OQ_THREADS, ring_tile(p.ebno_e1, eb_len, tile), OQ_SM_RING, &bars[b]);
                        bulk_g2s(t_e2 + b * OQ_T * OQ_THREADS, ring_tile(p.ebno_e2, eb_len, tile), OQ_SM_RING, &bars[b]);
                    }
                }
            };
            auto ring_store = [&](long long tile) {                   // write the (in-place updated) tile back to HBM
                const int b = (int)(tile % PP_NBUF);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    bulk_s2g(ring_tile(p.agc_ring, agc_len, tile), t_agc + b * OQ_T * OQ_THREADS, OQ_SM_RING);
                    if (ebno_on) {
                        bulk_s2g(ring_tile(p.ebno_e1, eb_len, tile), t_e1 + b * OQ_T * OQ_THREADS, OQ_SM_RING);
                        bulk_s2g(ring_tile(p.ebno_e2, eb_len, tile), t_e2 + b * OQ_T * OQ_THREADS, OQ_SM_RING);
                    }
                    bulk_commit();
                }
            };
            unsigned phases = 0u;
            long long rt = S / OQ_T;                                  // current ring tile
            bool ring_next_issued = false, ring_dirty = false;
            ring_load(rt);
            if ((rt + 1) * OQ_T < S_end) { ring_load(rt + 1); ring_next_issued = true; }
            PP_WAIT((int)(rt % PP_NBUF));
            for (int j = 0; j < nB; j++) {
                const int sl = j & 1;
                const int ro = (int)(S & (OQ_T - 1));
                const int rslot = (((int)(rt % PP_NBUF)) * OQ_T + ro) * OQ_THREADS + lane;   // this sample's slot in the staged ring tiles
                const double w41 = p.w41v[p41], w8 = p.w8v[p8];
                p41++; if (p41 > k41) p41 = 0;
                p8++; if (p8 > k8) p8 = 0;
                nb_sync(BAR_Z + sl);                           // Z_j: FIR output of this sample
                const double sre = HAND(sl, 0), sim = HAND(sl, 1);
                TR(2);
                const double dabval = sqrt(sre * sre + sim * sim);                // :461
                if (ebno_on) {                                                    // OQPSKEbNoMeasure::Update (DSP.cpp:729-744)
                    const double sq = dabval * dabval;
                    eb_sum2 = eb_sum2 - t_e2[rslot]; eb_sum2 = eb_sum2 + fabs(sq); t_e2[rslot] = fabs(sq);
                    eb_sum1 = eb_sum1 - t_e1[rslot]; eb_sum1 = eb_sum1 + fabs(dabval); t_e1[rslot] = fabs(dabval);
                    // read-out over the last OQ_EBNO_TAIL samples of the launch only (see oqpsk_demod.cu)
                    if (j >= eb_from_j) {
                        const double e2val = eb_sum2 / ((double)eb_len), mean = eb_sum1 / ((double)eb_len);
                        const double mean_sq = mean * mean;
                        double var = (e2val) - (mean * mean);
                        var -= (0.024709 * mean_sq);
                        double mvr = (((Fs * mean_sq / (2.0 * fbr * var))) * 0.13743);
                        if (mvr < 0.000000001) mvr = 0.000000001;
                        double tebno = 10.0 * log10(mvr);
                        if (isnan(tebno)) tebno = 50;
                        if (tebno > 50.0) tebno = 50;
                        if (tebno < 0.0) tebno = 0;
                        eb_ebno = eb_ebno * 0.8 + 0.2 * tebno;
                    }
                }
                {   // AGC::Update (DSP.cpp:370-379)
                    agc_sum = agc_sum - t_agc[rslot];
                    agc_sum = agc_sum + fabs(dabval);
                    t_agc[rslot] = fabs(dabval);
                    ring_dirty = true;
                    agc_val = div_fast(1.414213562, fmax(div_exact(agc_sum, (double)agc_len, r_agc), 0.000001));   // == the IEEE quotient (tools/micro/div_test.cu)
                    agc_val = fmax(agc_val, 0.000001);
                }
                double2 sig2 = make_double2(sre * agc_val, sim * agc_val);        // :466
                const double abval = hypot_fast(sig2.x, sig2.y);                  // :469 std::abs
                TR(10);
                if (abval > 2.84) { const double g = (2.84 / abval); sig2 = make_double2(g * sig2.x, g * sig2.y); }   // :470
                // ---- symbol timing, feed-forward part (:473-477)
                const double ab2 = abval * abval;
                const double st_diff = (0.0 * ab2 + (1.0 - 0.0) * dly_s0) - (ab2);    // Delay(1): weighting 0 -> x[n-1]
                dly_s0 = ab2;
                double st_d1out, st_d2out;
                {
                    const double older = (k41 == 3) ? d41_2 : (k41 == 2 ? d41_1 : d41_0);
                    const double newer = (k41 == 3) ? d41_1 : (k41 == 2 ? d41_0 : st_diff);
                    st_d1out = (w41 * newer + (1.0 - w41) * older);
                    d41_2 = d41_1; d41_1 = d41_0; d41_0 = st_diff;
                }
                {
                    const double older = (k41 == 3) ? d42_2 : (k41 == 2 ? d42_1 : d42_0);
                    const double newer = (k41 == 3) ? d42_1 : (k41 == 2 ? d42_0 : st_d1out);
                    st_d2out = (w41 * newer + (1.0 - w41) * older);
                    d42_2 = d42_1; d42_1 = d42_0; d42_0 = st_d1out;
                }
                double st_eta = (st_d2out - st_diff) * st_d1out;
                st_eta = biquad_update(res, st_eta, res_a1, res_a2, res_b0, res_b1, res_b2);
                double d8out;
                {
                    const double older = (k8 == 3) ? d8_2 : (k8 == 2 ? d8_1 : d8_0);
                    const double newer = (k8 == 3) ? d8_1 : (k8 == 2 ? d8_0 : st_eta);
                    d8out = (w8 * newer + (1.0 - w8) * older);
                    d8_2 = d8_1; d8_1 = d8_0; d8_0 = st_eta;
                }
                // slot sl's fields were last read by T(j-2) and K(j-2), which precede X_{j-1} -> Z_j: free
                HAND(sl, 2) = sig2.x; HAND(sl, 3) = sig2.y; HAND(sl, 4) = st_eta; HAND(sl, 5) = d8out;
                PP_HANDOFF_FENCE();
                nb_arrive(BAR_YT + sl);                        // timing inputs -> warp T
                nb_arrive(BAR_YK + sl);                        // sig2 -> warp K
                TR(3);
                // ---- ring tile bookkeeping (warp-uniform)
                S++;
                if ((S & (OQ_T - 1)) == 0) {
                    ring_store(rt);                                   // the finished tile goes back to HBM
                    ring_dirty = false;
                    rt++;
                    if (S < S_end) {
                        PP_WAIT((int)(rt % PP_NBUF));                 // next tile (requested a tile ago)
                        ring_next_issued = false;
                        if ((rt + 1) * OQ_T < S_end) {
                            // the buffer being refilled was stored a whole tile ago: only the store committed just now may still
                            // be reading shared memory
                            bulk_wait_read_1();
                            ring_load(rt + 1); ring_next_issued = true;
                        }
                    }
                }
            }
            if (ring_dirty) ring_store(rt);
            if (ring_next_issued) PP_WAIT((int)((rt + 1) % PP_NBUF));
            bulk_wait_all();
        }
        LD(D_AGC_SUM) = agc_sum; LD(D_AGC_VAL) = agc_val;
        LD(D_EB_SUM1) = eb_sum1; LD(D_EB_SUM2) = eb_sum2; LD(D_EB_EBNO) = eb_ebno;
        LD(D_DLY_S0) = dly_s0;
        LD(D_DLY41_0) = d41_0; LD(D_DLY41_1) = d41_1; LD(D_DLY41_2) = d41_2;
        LD(D_DLY42_0) = d42_0; LD(D_DLY42_1) = d42_1; LD(D_DLY42_2) = d42_2;
        LD(D_DLY8_0) = d8_0; LD(D_DLY8_1) = d8_1; LD(D_DLY8_2) = d8_2;
        LD(D_RES_X1) = res.x1; LD(D_RES_X2) = res.x2; LD(D_RES_Y1) = res.y1; LD(D_RES_Y2) = res.y2;
    }
    // ======================================================================================= warp F: matched filter
    else if (warp == 0) {
        for (int k = 0; k < OQ_NT1; k++) {
            const double vr = p.fir_re[(size_t)k * cpad + ch], vi = p.fir_im[(size_t)k * cpad + ch];
            s_re[k * OQ_THREADS + lane] = vr; s_re[(k + OQ_NT1) * OQ_THREADS + lane] = vr;
            s_im[k * OQ_THREADS + lane] = vi; s_im[(k + OQ_NT1) * OQ_THREADS + lane] = vi;
        }
        __syncthreads();                                       // (1)
        // output j (:456) = sum over the 55 mixed samples older than sample i0+j; the newest of them (slot `tail`) is produced
        // by warp K2 one sample earlier, the 54 older terms are summed ahead of that
        int tail = (int)((S0 + OQ_NT1 - 1) % OQ_NT1);
        double nfre = 0, nfim = 0;
        if (nB > 0) fir54(p, s_re + (tail + 2) * OQ_THREADS + lane, s_im + (tail + 2) * OQ_THREADS + lane, nfre, nfim);
        for (int j = 0; j < nB; j++) {
            const int sl = j & 1;
            if (j > 0) nb_sync(BAR_X + ((j - 1) & 1));        // X_{j-1}
            TR(0);
            nfre += p.taps[54] * s_re[tail * OQ_THREADS + lane]; nfim += p.taps[54] * s_im[tail * OQ_THREADS + lane];
            // slot sl's F->E fields were read by E(j-2), before X_{j-1}: free
            HAND(sl, 0) = nfre; HAND(sl, 1) = nfim;
            PP_HANDOFF_FENCE();
            nb_arrive(BAR_Z + sl);                             // Z_j
            TR(1);
            tail++; if (tail >= OQ_NT1) tail = 0;
            if (j + 1 < nB) fir54(p, s_re + (tail + 2) * OQ_THREADS + lane, s_im + (tail + 2) * OQ_THREADS + lane, nfre, nfim);
        }
        if (nB > 0) nb_sync(BAR_X + ((nB - 1) & 1));          // X_{nB-1}: pair the last arrival of warp K2
    }
    // ======================================================================================= warp A: input + coarse-estimator ring
    else {
        const int16_t *row = pcm + (size_t)ch * stride;
        // PCM: each lane reads its own channel row 8 samples (16 bytes) at a time with plain vector loads, one block ahead of use
        // (rows are 16-byte aligned and a multiple of 8 samples long: host-checked). The bulk-copy tiles used before cost 32
        // serialised copy instructions per 32 samples (one per lane) for 64 bytes each.
        const int4 *row4 = reinterpret_cast<const int4 *>(row);
        auto ld_blk = [&](int blk) -> int4 {
            return (live && (long long)blk * 8 < (long long)stride) ? __ldg(row4 + blk) : make_int4(0, 0, 0, 0);
        };
        int pk_blk = a.i0 >> 3;
        int4 pk = ld_blk(pk_blk), pk_next = ld_blk(pk_blk + 1);   // 8 consecutive PCM samples of this lane's channel, and the next 8
        auto dval_at = [&](int ii) -> double {                    // ((double)*ptr)/32768.0 (:390); ii advances by one per call
            if ((ii >> 3) != pk_blk) { pk_blk = ii >> 3; pk = pk_next; pk_next = ld_blk(pk_blk + 1); }
            const int k = ii & 7;
            const int w = (k < 2) ? pk.x : (k < 4) ? pk.y : (k < 6) ? pk.z : pk.w;
            int v = (k & 1) ? (w >> 16) : (int)(short)(w & 0xffff);
            if (!live) v = 0;
            return ((double)v) / 32768.0;
        };
        __syncthreads();                                       // (1) the slot may have re-centred mixer_center
        Osc mc = {LD(D_MC_PTR), LD(D_MC_STEP), LD(D_MC_FREQ), LD(D_MC_LAST)};
        Osc sr = {LD(D_SR_PTR), LD(D_SR_STEP), LD(D_SR_FREQ), LD(D_SR_LAST)};   // st_osc_ref (:603): nothing in the loop reads its pointer
        int bb_pos = a.bb_pos, coarse_counter = a.coarse_counter;
        double2 *bb_row = p.bb + (size_t)ch * p.bb_len;
        const int bbn = p.bb_len;                               // a multiple of 8
        const bool cpu_reduce = p.cpu_reduce != 0;
        double cc_re, cc_im;
        { const int t = osc_index(mc.ptr); cc_re = __ldcg(cos_t + t); cc_im = __ldcg(sin_t + t); }
        // This warp runs ahead of the demodulator loop: nothing it computes depends on the loop (PCM, mixer_center, the estimator
        // ring). It decodes the input into a two-tile ring for warp K2 and writes the estimator ring one full 128-byte line (8
        // samples) per lane at a time, so that every 32-byte sector reaches HBM whole.
        const int n = a.i1 - a.i0;
        unsigned aph = 0u;                                      // parities of the two input-tile-empty mbarriers
        int line_first = bb_pos & 7;                            // entries of the open line below this index were written by an earlier launch
        for (int e = 0; e < n; e++) {
            const int tb = (e >> 5) & 1;
            if ((e & 31) == 0 && e >= PP_DV) { mbar_wait_relaxed(&bars[7 + tb], (aph >> tb) & 1u); aph ^= (1u << tb); }
            const double dcur = dval_at(a.i0 + e);
            dv[(e & (PP_DV - 1)) * 32 + lane] = dcur;
            // ---- A: coarse-estimator ring (:410-429); the host ends the segment on the trigger sample
            if (!(e == 0 && a.skip_a_first)) {
                if (coarse_counter >= Fs || !cpu_reduce) {
                    bbst[(bb_pos & 7) * 32 + lane] = make_double2(cc_re * dcur, cc_im * dcur);
                    if ((bb_pos & 7) == 7) {
                        if (live) for (int k = line_first; k < 8; k++) bb_row[(bb_pos & ~7) + k] = bbst[k * 32 + lane];
                        line_first = 0;
                    }
                    bb_pos++; if (bb_pos >= bbn) bb_pos = 0;
                }
            }
            if (!(e == n - 1 && a.stop_after_a)) {
                coarse_counter++;                                                 // :431
                osc_next_frame(mc);                                               // :601
                osc_next_frame(sr);                                               // :603
                { const int t = osc_index(mc.ptr); cc_re = __ldcg(cos_t + t); cc_im = __ldcg(sin_t + t); }   // L2 only: L1 is kept for warp T's entries
            }
            if ((e & 31) == 31 || e == n - 1)
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bars[3 + tb])) : "memory");   // tile (or the rest) complete
        }
        if (live) for (int k = line_first; k < (bb_pos & 7); k++) bb_row[(bb_pos & ~7) + k] = bbst[k * 32 + lane];   // the open line
        LD(D_MC_PTR) = mc.ptr; LD(D_MC_STEP) = mc.step; LD(D_MC_FREQ) = mc.freq; LD(D_MC_LAST) = mc.last;
        LD(D_SR_PTR) = sr.ptr; LD(D_SR_LAST) = sr.last;
    }
    __syncthreads();                                           // (2) every warp is done with the FIR window
    for (int k = (int)(threadIdx.x >> 5); k < OQ_NT1; k += (int)(blockDim.x >> 5)) {
        p.fir_re[(size_t)k * cpad + ch] = s_re[k * OQ_THREADS + lane];
        p.fir_im[(size_t)k * cpad + ch] = s_im[k * OQ_THREADS + lane];
    }
#undef HAND
}

int oqpsk_pipe_launch(const DemodParams &p, const SegmentArgs &a, const int16_t *d_pcm, size_t stride, cudaStream_t s)
{
    const int grid = (p.n_channels + OQ_THREADS - 1) / OQ_THREADS;
    const size_t smem = (size_t)PP_SM_TOTAL;
    JB_CUDA(cudaFuncSetAttribute(oqpsk_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    oqpsk_pipe_kernel<<<grid, PP_THREADS, smem, s>>>(p, a, d_pcm, stride);
    JB_CUDA(cudaGetLastError());
    return 0;
}

#undef LD
#undef LI
} // namespace jb

#undef PP_WAIT
#undef TR
