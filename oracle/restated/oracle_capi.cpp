// TEST INFRASTRUCTURE ONLY (oracle): extern "C" surface of the CPU restatement for ctypes.
#include "demod_oracle.h"
#include "fec_oracle.h"
#include "burst_oracle.h"
#include <cstring>
using namespace jor;

struct OrHandle { int kind; OqpskDemodOracle *oq; MskDemodOracle *msk; BurstMskOracle *bmsk; BurstOqpskOracle *boq; };

extern "C" {
void *jor_demod_new(int kind, double fb, double Fs, double freq_center, double lockingbw, int fft_power,
                    double signalthreshold, int afc, int sql, int cpureduce)
{
    DemodSettings s; s.coarsefreqest_fft_power = fft_power; s.freq_center = freq_center; s.lockingbw = lockingbw;
    s.fb = fb; s.Fs = Fs; s.signalthreshold = signalthreshold; s.afc = afc; s.sql = sql; s.cpuReduce = cpureduce;
    OrHandle *h = new OrHandle(); h->kind = kind; h->oq = 0; h->msk = 0; h->bmsk = 0; h->boq = 0;
    if (kind == 0) h->oq = new OqpskDemodOracle(s); else h->msk = new MskDemodOracle(s);
    return h;
}
void *jor_burst_msk_new(double fb, double Fs, double freq_center, double lockingbw, double signalthreshold)
{ OrHandle *h = new OrHandle(); h->kind = 2; h->oq = 0; h->msk = 0; h->boq = 0; h->bmsk = new BurstMskOracle(fb, Fs, freq_center, lockingbw, signalthreshold); return h; }
void *jor_burst_oqpsk_new(double fb, double Fs, double freq_center, double lockingbw, double signalthreshold)
{ OrHandle *h = new OrHandle(); h->kind = 3; h->oq = 0; h->msk = 0; h->bmsk = 0; h->boq = new BurstOqpskOracle(fb, Fs, freq_center, lockingbw, signalthreshold); return h; }
void jor_write(void *hv, const int16_t *pcm, long n)
{ OrHandle *h = (OrHandle *)hv; if (h->kind == 0) h->oq->writeData(pcm, n); else if (h->kind == 1) h->msk->writeData(pcm, n); else if (h->kind == 2) h->bmsk->writeData(pcm, n); else h->boq->writeData(pcm, n); }
void jor_set_dcd(void *hv, int d)
{ OrHandle *h = (OrHandle *)hv; if (h->kind == 0) h->oq->DCDstatSlot(d != 0); else if (h->kind == 1) h->msk->DCDstatSlot(d != 0); else if (h->kind == 2) h->bmsk->dcd = (d != 0); }
static std::vector<short> &soft_of(OrHandle *h) { return h->kind == 0 ? h->oq->soft_out : (h->kind == 1 ? h->msk->soft_out : (h->kind == 2 ? h->bmsk->soft_out : h->boq->soft_out)); }
long jor_soft_count(void *hv)
{ OrHandle *h = (OrHandle *)hv; return (long)soft_of(h).size(); }
long jor_aux_take(void *hv, int which, double *out, long cap)     // burst: 0 = EbNo per burst, 1 = trident log (5 values per test)
{
    OrHandle *h = (OrHandle *)hv; if (h->kind < 2) return 0;
    std::vector<double> &v = h->kind == 2 ? (which == 0 ? h->bmsk->ebno_log : h->bmsk->trident_log) : (which == 0 ? h->boq->ebno_log : h->boq->trident_log);
    long n = (long)v.size(); if (n > cap) n = cap;
    memcpy(out, v.data(), n * sizeof(double)); v.erase(v.begin(), v.begin() + n); return n;
}
long jor_soft_take(void *hv, short *out, long cap)
{
    OrHandle *h = (OrHandle *)hv; std::vector<short> &v = soft_of(h);
    long n = (long)v.size(); if (n > cap) n = cap;
    memcpy(out, v.data(), n * sizeof(short)); v.erase(v.begin(), v.begin() + n); return n;
}
long jor_cfe_log_take(void *hv, double *out, long cap)
{
    OrHandle *h = (OrHandle *)hv; if (h->kind >= 2) return 0;
    std::vector<double> &v = h->kind == 0 ? h->oq->cfe_log : h->msk->cfe_log;
    long n = (long)v.size(); if (n > cap) n = cap;
    memcpy(out, v.data(), n * sizeof(double)); v.erase(v.begin(), v.begin() + n); return n;
}
// same layout as jref_state (oracle/ref_driver.cpp)
int jor_state(void *hv, double *o)
{
    OrHandle *h = (OrHandle *)hv;
    if (h->kind == 0) {
        OqpskDemodOracle *d = h->oq;
        o[0] = d->mixer2.freq; o[1] = d->mixer2.WTptr; o[2] = d->mixer_center.freq; o[3] = d->st_osc.freq; o[4] = d->st_osc.WTptr;
        o[5] = d->agc.AGCVal; o[6] = d->mse; o[7] = d->ebno.EbNo; o[8] = d->marg.Val; o[9] = d->cfe.freq_offset_est;
        o[10] = (double)d->n_sig_true; o[11] = (double)d->n_sig_false; o[12] = d->mixer_center.WTptr; o[13] = d->st_osc_ref.WTptr;
    } else if (h->kind == 3) {
        BurstOqpskOracle *d = h->boq;
        o[0] = d->mixer2.freq; o[1] = d->mixer2.WTptr; o[2] = d->mixer2.freq; o[3] = d->st_osc.freq; o[4] = d->st_osc.WTptr;
        o[5] = d->agc.AGCVal; o[6] = d->mse; o[7] = d->ebno.EbNo; o[8] = d->vol_gain; o[9] = d->rotator_freq;
        o[10] = (double)d->n_sig_true; o[11] = (double)d->n_sig_false; o[12] = (double)d->cntr; o[13] = (double)d->startstop;
    } else if (h->kind == 2) {
        BurstMskOracle *d = h->bmsk;      // same layout as jref_state for burst kinds
        o[0] = d->mixer2.freq; o[1] = d->mixer2.WTptr; o[2] = d->mixer_center.freq; o[3] = d->st_osc.freq; o[4] = d->st_osc.WTptr;
        o[5] = d->agc.AGCVal; o[6] = d->mse; o[7] = d->ebno.EbNo; o[8] = d->vol_gain; o[9] = d->rotator_freq;
        o[10] = (double)d->n_sig_true; o[11] = (double)d->n_sig_false; o[12] = (double)d->cntr; o[13] = (double)d->startstop;
    } else {
        MskDemodOracle *d = h->msk;
        o[0] = d->mixer2.freq; o[1] = d->mixer2.WTptr; o[2] = d->mixer_center.freq; o[3] = d->st_osc.freq; o[4] = d->st_osc.WTptr;
        o[5] = d->agc.AGCVal; o[6] = d->mse; o[7] = d->ebno.EbNo; o[8] = d->marg.Val; o[9] = d->cfe.freq_offset_est;
        o[10] = (double)d->n_sig_true; o[11] = (double)d->n_sig_false; o[12] = d->mixer_center.WTptr; o[13] = 0;
    }
    return 14;
}
void jor_free(void *hv) { OrHandle *h = (OrHandle *)hv; delete h->oq; delete h->msk; delete h->bmsk; delete h->boq; delete h; }

int jor_rrc_design(double alpha, int firsize, double Fs, double symbol_freq, double *out, int cap)
{ std::vector<double> p = rrc_design(alpha, firsize, Fs, symbol_freq); int n = (int)p.size(); for (int i = 0; i < n && i < cap; i++) out[i] = p[i]; return n; }
// restated JFastFir over a restated RRC kernel, configured as jref_jfastfir_rrc (oracle/ref_driver.cpp)
void jor_jfastfir_rrc(double alpha, int firsize, double Fs, double symbol_freq, int nfft, double *inout_ri, long n)
{
    std::vector<double> pts = rrc_design(alpha, firsize, Fs, symbol_freq);
    QVector<double> qp((int)pts.size());
    for (size_t i = 0; i < pts.size(); i++) qp[(int)i] = pts[i];
    JFastFir fir; fir.SetKernel(qp, nfft);
    std::vector<JFastFir::cpx_type> v(n);
    for (long i = 0; i < n; i++) v[i] = JFastFir::cpx_type(inout_ri[2 * i], inout_ri[2 * i + 1]);
    fir.update(v.data(), (int)n);
    for (long i = 0; i < n; i++) { inout_ri[2 * i] = v[i].real(); inout_ri[2 * i + 1] = v[i].imag(); }
}
void jor_trig_tables(double *s, double *c) { for (int i = 0; i < WTSIZE; i++) { s[i] = trig().SinWT[i]; c[i] = trig().CosWT[i]; } }
int jor_qround(double d) { return jor::qRound(d); }
void jor_fft(int n, int inverse, const double *in_ri, double *out_ri)
{ std::vector<cpx> x(n); for (int i = 0; i < n; i++) x[i] = cpx(in_ri[2 * i], in_ri[2 * i + 1]); fft_pow2(x.data(), n, inverse != 0);
  for (int i = 0; i < n; i++) { out_ri[2 * i] = x[i].real(); out_ri[2 * i + 1] = x[i].imag(); } }

void *jor_cfe_new(int power, double lockingbw, double fb, double Fs) { CoarseFreqEstimate *c = new CoarseFreqEstimate(); c->setSettings(power, lockingbw, fb, Fs); return c; }
double jor_cfe_process(void *cv, const double *ri, double *y_out, double *raw_est)
{
    CoarseFreqEstimate *c = (CoarseFreqEstimate *)cv; std::vector<cpx> d(c->nfft);
    for (int i = 0; i < c->nfft; i++) d[i] = cpx(ri[2 * i], ri[2 * i + 1]);
    double e = c->ProcessBasebandData(d);
    if (y_out) for (int i = 0; i < c->nfft; i++) y_out[i] = c->y[i];
    if (raw_est) *raw_est = c->freq_offset_est;
    return e;
}
void jor_cfe_bigchange(void *cv) { ((CoarseFreqEstimate *)cv)->bigchange(); }
void jor_cfe_free(void *cv) { delete (CoarseFreqEstimate *)cv; }

// ---- FEC ----
void jor_deinterleave(const int *block, int cols, uint8_t *out) { oracle_deinterleave(block, cols, out); }
void *jor_viterbi_new(int pad) { return new ContinuousViterbiOracle(pad); }
int jor_viterbi_decode_continuous(void *v, const uint8_t *soft, int n, int *bits)
{ std::vector<int> r = ((ContinuousViterbiOracle *)v)->decode(soft, n); for (size_t i = 0; i < r.size(); i++) bits[i] = r[i]; return (int)r.size(); }
void jor_viterbi_free(void *v) { delete (ContinuousViterbiOracle *)v; }
// raw libcorrect-restated entry points for block tests
int jor_conv_decode_soft(const uint8_t *soft, int nbits, uint8_t *msg)
{ correct_convolutional_polynomial_t poly[2] = {109, 79}; correct_convolutional *c = correct_convolutional_create(2, 7, poly);
  int r = (int)correct_convolutional_decode_soft(c, soft, nbits, msg); correct_convolutional_destroy(c); return r; }
int jor_conv_encode(const uint8_t *msg, int msg_len, uint8_t *enc)
{ correct_convolutional_polynomial_t poly[2] = {109, 79}; correct_convolutional *c = correct_convolutional_create(2, 7, poly);
  int r = (int)correct_convolutional_encode(c, msg, msg_len, enc); correct_convolutional_destroy(c); return r; }

void *jor_pchan_new(int fb) { return new PChannelOracle(fb); }
void jor_pchan_lost_signal(void *p) { ((PChannelOracle *)p)->lostSignal(); }
// The reference's direct connections between one continuous demodulator and one AeroL (JAERO/mainwindow.cpp:198-199,234,237,432,508):
// every emitted soft-bit vector is decoded at once and the resulting DataCarrierDetect state is back in the demodulator before its
// next sample; SignalStatus(false) is AeroL::LostSignal.
struct WireCtx { OrHandle *d; PChannelOracle *p; };
static void wire_set_dcd(WireCtx *w) { if (w->d->kind == 0) w->d->oq->DCDstatSlot(w->p->datacd); else w->d->msk->DCDstatSlot(w->p->datacd); }
static void wire_emit(void *ctx, const short *bits, int n) { WireCtx *w = (WireCtx *)ctx; w->p->process(bits, n); wire_set_dcd(w); }
static void wire_sigstat(void *ctx, bool ok) { WireCtx *w = (WireCtx *)ctx; if (!ok) { w->p->lostSignal(); wire_set_dcd(w); } }
void jor_wire_pchan(void *hv, void *pv)
{
    OrHandle *h = (OrHandle *)hv; WireCtx *w = new WireCtx{h, (PChannelOracle *)pv};   // lives as long as the test process
    if (h->kind == 0) { h->oq->on_emit = wire_emit; h->oq->on_sigstat = wire_sigstat; h->oq->hook_ctx = w; }
    else if (h->kind == 1) { h->msk->on_emit = wire_emit; h->msk->on_sigstat = wire_sigstat; h->msk->hook_ctx = w; }
}
void jor_pchan_process(void *p, const short *soft, int n) { ((PChannelOracle *)p)->process(soft, n); }
void jor_pchan_update_dcd(void *p) { ((PChannelOracle *)p)->updateDCD(); }
int jor_pchan_dcd(void *p) { return ((PChannelOracle *)p)->datacd ? 1 : 0; }
long jor_pchan_su_count(void *p) { return (long)((PChannelOracle *)p)->sus.size(); }
long jor_pchan_su_take(void *p, uint8_t *bytes12, int *crc_ok, long *frame, long cap)
{
    PChannelOracle *o = (PChannelOracle *)p; long n = (long)o->sus.size(); if (n > cap) n = cap;
    for (long i = 0; i < n; i++) { memcpy(bytes12 + 12 * i, o->sus[i].bytes, 12); crc_ok[i] = o->sus[i].crc_ok; frame[i] = o->sus[i].frame; }
    o->sus.erase(o->sus.begin(), o->sus.begin() + n); return n;
}
void jor_pchan_free(void *p) { delete (PChannelOracle *)p; }
// ---- C channel (8400)
void *jor_cchan_new() { return new CChannelOracle(); }
void jor_cchan_process(void *p, const short *soft, int n) { ((CChannelOracle *)p)->process(soft, n); }
void jor_cchan_update_dcd(void *p) { ((CChannelOracle *)p)->updateDCD(); }
int jor_cchan_dcd(void *p) { return ((CChannelOracle *)p)->datacd ? 1 : 0; }
long jor_cchan_frame_count(void *p) { return (long)((CChannelOracle *)p)->frames.size(); }
// frames: su [n][3][12], crc_ok [n][3], voice [n][300]
long jor_cchan_take(void *p, uint8_t *su, int *crc_ok, uint8_t *voice, long cap)
{
    CChannelOracle *o = (CChannelOracle *)p;
    long n = (long)o->frames.size(); if (n > cap) n = cap;
    for (long k = 0; k < n; k++) {
        for (int q = 0; q < 3; q++) { for (int b = 0; b < 12; b++) su[(k * 3 + q) * 12 + b] = o->frames[k].su[q].bytes[b]; crc_ok[k * 3 + q] = o->frames[k].su[q].crc_ok; }
        for (int b = 0; b < 300; b++) voice[k * 300 + b] = o->frames[k].voice[b];
    }
    o->frames.erase(o->frames.begin(), o->frames.begin() + n);
    return n;
}
void jor_cchan_free(void *p) { delete (CChannelOracle *)p; }
// ---- R/T burst channel
void *jor_rt_new(int fb) { return new RTChannelOracle(fb); }
void jor_rt_process(void *p, const short *soft, int n, int vector_semantics) { ((RTChannelOracle *)p)->process(soft, n, vector_semantics != 0); }
void jor_rt_update_dcd(void *p) { ((RTChannelOracle *)p)->updateDCD(); }
long jor_rt_packet_count(void *p) { return (long)((RTChannelOracle *)p)->packets.size(); }
long jor_rt_trials(void *p) { return ((RTChannelOracle *)p)->n_trials; }
// packet k: returns length, fills type / nsus / bit_index
int jor_rt_packet(void *p, long k, int *type, int *nsus, long *bit_index, uint8_t *bytes, int cap)
{
    RTChannelOracle *o = (RTChannelOracle *)p;
    if (k < 0 || k >= (long)o->packets.size()) return -1;
    const RTPacket &pk = o->packets[k];
    *type = pk.type; *nsus = pk.nsus; *bit_index = pk.bit_index;
    const int n = (int)pk.bytes.size() < cap ? (int)pk.bytes.size() : cap;
    for (int i = 0; i < n; i++) bytes[i] = pk.bytes[i];
    return (int)pk.bytes.size();
}
void jor_rt_free(void *p) { delete (RTChannelOracle *)p; }
uint16_t jor_crc16(const uint8_t *b, int n) { return oracle_crc16(b, n); }
}
