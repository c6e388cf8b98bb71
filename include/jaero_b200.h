/* jaero_b200 — C ABI of the B200-native JAERO demodulator / Viterbi hot path.
 *
 * Drop-in boundary (SURVEY.md §8b). Every entry point below replaces a piece of the reference's
 * per-instance C++/Qt interface with a *batched* call over many independent channels; a single
 * reference object is a batch of one. Plain pointers and sizes only — no Qt, no torch, no CUDA
 * types. All functions return 0 on success or a negative JAERO_E_* code; jaero_last_error()
 * gives the message for the calling thread. There is NO CPU fallback: if no CUDA device is
 * usable the create calls fail with JAERO_E_CUDA.
 *
 *   reference interface (file:line)                               this header
 *   -------------------------------------------------------------  ---------------------------
 *   OqpskDemodulator::Settings  JAERO/oqpskdemodulator.h:20-39      jaero_settings
 *   MskDemodulator::Settings    JAERO/mskdemodulator.h:24-45        jaero_settings
 *   ctor + setSettings + setAFC/setSQL/setCPUReduce + start()
 *     JAERO/oqpskdemodulator.cpp:8-117,149-163,175-289,312-315      jaero_batch_create
 *     JAERO/mskdemodulator.cpp:9-84,105-118,135-263,296-299
 *   qint64 writeData(const char*, qint64)
 *     JAERO/oqpskdemodulator.cpp:334-627, mskdemodulator.cpp:313-488 jaero_batch_write[_device]
 *   signal processDemodulatedSoftBits(const QVector<short>&)
 *     JAERO/oqpskdemodulator.h:67, mskdemodulator.h:152             jaero_batch_read_softbits
 *   slot DCDstatSlot(bool)  oqpskdemodulator.cpp:679-684            jaero_batch_set_dcd
 *   slot CenterFreqChangedSlot(double) oqpskdemodulator.cpp:291-310 jaero_batch_set_center_freq
 *   signals MSESignal / EbNoMeasurmentSignal / SignalStatus / Plottables,
 *     getCurrentFreq()  oqpskdemodulator.cpp:322-325,670-675         jaero_batch_get_status
 *   CoarseFreqEstimate::ProcessBasebandData + FreqOffsetEstimateSlot
 *     JAERO/coarsefreqestimate.cpp:90-137, oqpskdemodulator.cpp:629-677   (inside jaero_batch_write)
 *   AeroLInterleaver::deinterleave_ba  JAERO/aerol.cpp:603-625       jaero_viterbi_decode_continuous(cols>0)
 *   JConvolutionalCodec::SetCode / Decode_Continuous / Decode_soft
 *     JAERO/jconvolutionalcodec.cpp:20-29,151-201,98-125            jaero_viterbi_*
 *   destructor                                                      jaero_batch_destroy / jaero_viterbi_destroy
 */
#ifndef JAERO_B200_H
#define JAERO_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define JAERO_OK 0
#define JAERO_E_ARG (-1)      /* bad argument */
#define JAERO_E_CUDA (-2)     /* CUDA runtime error / no device (no CPU fallback exists) */
#define JAERO_E_STATE (-3)    /* call not valid in this state */
#define JAERO_E_OVERFLOW (-4) /* a soft-bit ring overflowed because the caller did not drain it */

#define JAERO_KIND_OQPSK 0 /* continuous 8400/10500 bps OQPSK, JAERO/oqpskdemodulator.cpp */
#define JAERO_KIND_MSK 1   /* continuous 600/1200 bps MSK,     JAERO/mskdemodulator.cpp */

/* Same fields, defaults and units as the reference's Settings structs. */
typedef struct jaero_settings {
    int kind;                    /* JAERO_KIND_* */
    int coarsefreqest_fft_power; /* 14 (OQPSK) / 13 (MSK) */
    double freq_center;          /* Hz; used for every channel unless per-channel values are given */
    double lockingbw;            /* Hz */
    double fb;                   /* bits/s: 600, 1200, 8400, 10500 */
    double Fs;                   /* Hz, 48000 */
    double signalthreshold;      /* 0.65 (OQPSK) / 0.5 (MSK) */
    int afc;                     /* setAFC */
    int sql;                     /* setSQL */
    int cpu_reduce;              /* setCPUReduce */
    int report_ebno;             /* 1: keep the two 2 s EbNo moving averages (observable only) */
} jaero_settings;

/* Per-channel telemetry: what the reference emits as MSESignal, EbNoMeasurmentSignal,
 * SignalStatus, Plottables(freq_est, freq_center, bw) plus the loop state used by parity tests. */
typedef struct jaero_status {
    double mixer2_freq;   /* Hz  (Plottables freq_est) */
    double mixer2_wtptr;  /* NCO table pointer [0,19999) */
    double center_freq;   /* Hz  (getCurrentFreq) */
    double st_freq;       /* symbol-timing oscillator Hz */
    double st_wtptr;
    double agc;           /* AGC::AGCVal */
    double mse;           /* MSESignal */
    double ebno;          /* EbNoMeasurmentSignal (0 if report_ebno==0) */
    double marg;          /* residual-bias moving average */
    double cfe_est;       /* last coarse frequency estimate (Hz offset) */
    double n_sig_true;    /* SignalStatus(true) count */
    double n_sig_false;   /* SignalStatus(false) count */
    double center_wtptr;
    double st_ref_wtptr;
    int64_t samples;      /* samples consumed so far */
    int64_t softbits;     /* soft values emitted so far (drained + still in the ring; burst markers included) */
    int32_t dcd;
    int32_t reserved;
    double peak_volume;   /* PeakVolume (oqpskdemodulator.cpp:393-405): max |input sample| / 32768 since the previous status read */
    double scatter[4];    /* ScatterPoints, decimated: the two most recent constellation points (re, im, re, im) as pointbuff holds them */
} jaero_status;

typedef struct jaero_batch jaero_batch;
typedef struct jaero_viterbi jaero_viterbi;

const char *jaero_last_error(void);
int jaero_device_count(void);

/* n_channels independent demodulators of one mode on one GPU. freq_center_per_channel may be NULL. */
int jaero_batch_create(const jaero_settings *settings, int n_channels,
                       const double *freq_center_per_channel, int device_ordinal, jaero_batch **out);
void jaero_batch_destroy(jaero_batch *b);
int jaero_batch_channels(const jaero_batch *b);

/* writeData for every channel: pcm[ch*channel_stride + i], i < n_samples, little-endian int16 mono,
 * HOST memory (the call stages it to the GPU). Asynchronous with respect to the host unless
 * followed by a read/status call; ordering between calls is preserved. */
int jaero_batch_write(jaero_batch *b, const int16_t *pcm, size_t n_samples, size_t channel_stride);
/* Same, pcm already resident in this GPU's memory (device pointer). */
int jaero_batch_write_device(jaero_batch *b, const int16_t *d_pcm, size_t n_samples, size_t channel_stride);
/* Block until everything queued so far has executed. */
int jaero_batch_sync(jaero_batch *b);

/* Drain the soft bits emitted since the last read (the concatenated payloads of the reference's
 * processDemodulatedSoftBits emits: multiples of 32 (OQPSK) / 12 (MSK) values 0..255).
 * out[ch*cap + k]; counts[ch] = number written for that channel. HOST pointers. */
int jaero_batch_read_softbits(jaero_batch *b, int16_t *out, size_t cap_per_channel, int32_t *counts);
/* Device-resident view of the same rings for on-GPU consumers (d_soft[ch*ring_cap + k], d_counts[ch]);
 * valid until the next write. jaero_batch_reset_softbits() marks them consumed. */
int jaero_batch_softbits_device(jaero_batch *b, const int16_t **d_soft, const int32_t **d_counts, size_t *ring_cap);
int jaero_batch_reset_softbits(jaero_batch *b);

int jaero_batch_set_dcd(jaero_batch *b, int channel, int dcd);            /* channel<0: all */
int jaero_batch_set_center_freq(jaero_batch *b, int channel, double hz);  /* CenterFreqChangedSlot */
/* setAFC / setSQL / setCPUReduce of the reference classes: every channel of the batch, effective from the next write */
int jaero_batch_set_afc(jaero_batch *b, int state);
int jaero_batch_set_sql(jaero_batch *b, int state);
int jaero_batch_set_cpu_reduce(jaero_batch *b, int state);
/* Seating of the channels inside the 10500 bps kernel. Channels never interact, so results do not depend on it; throughput does:
 * the library seats channels with the same symbol-timing phase next to each other (automatically, every JAERO_REGROUP_EPOCHS
 * estimator epochs; this call does it now when slot_of is NULL, or installs the given permutation slot_of[channel] = seat). */
int jaero_batch_regroup(jaero_batch *b, const int32_t *slot_of);
/* connect(demodulator, SIGNAL(SignalStatus(bool)), aerol, SLOT(SignalStatusSlot(bool))) (JAERO/mainwindow.cpp:432,508): with it, a
 * SignalStatus(false) clears the channel's DCD in the kernel and is handed to the device frame layer (jaero_pchannel_process_batch /
 * jaero_cchannel_process_batch) as a LostSignal at its soft-bit position. Off by default (host-driven DCD via jaero_batch_set_dcd). */
int jaero_batch_wire_signal_status(jaero_batch *b, int enabled);
int jaero_batch_get_status(jaero_batch *b, int channel, jaero_status *out);
int jaero_batch_get_status_all(jaero_batch *b, jaero_status *out /* [n_channels] */);
/* kernel launches issued by this batch so far (for bench.py's gpu_launches) */
int64_t jaero_batch_launch_count(const jaero_batch *b);
/* Run on a caller-owned CUDA stream (a cudaStream_t passed as void*; NULL = back to the batch's own stream),
 * so the caller's events / other work order against the demodulator kernels. */
int jaero_batch_set_stream(jaero_batch *b, void *cuda_stream);
/* Measurement aid: when enabled, every segment-kernel launch and every coarse-estimator run is bracketed by CUDA
 * events on the launch stream; get_profile() synchronises and returns the accumulated device milliseconds and
 * launch counts since the last call: out[0]=segment ms, out[1]=segment launches, out[2]=estimator ms,
 * out[3]=estimator runs, out[4]=samples per channel covered by the segment launches. */
int jaero_batch_set_profiling(jaero_batch *b, int enabled);
int jaero_batch_get_profile(jaero_batch *b, double out[5]);

/* ---- K=7 r=1/2 soft Viterbi (polys 109,79), one independent decoder per channel ---- */
int jaero_viterbi_create(int n_channels, int paddinglength, int device_ordinal, jaero_viterbi **out);
void jaero_viterbi_destroy(jaero_viterbi *v);
/* Decode_Continuous for every channel: soft[ch*n_soft + k] (0..255, 128 = erasure), n_soft even.
 * interleaver_cols > 0: soft is the *interleaved* 64 x cols block and the de-interleave gather
 * (AeroLInterleaver::deinterleave_ba) is fused in front; 0: soft is already in code order.
 * bits_out[ch*(n_soft/2) + k] in {0,1}. The 62-value overlap is carried per channel. HOST pointers.
 * n_valid[ch] (may be NULL) = number of bits Decode_Continuous returns for that channel: n_soft/2,
 * except on a channel's first call after create/reset, where QVector::mid() truncates the result to
 * n_soft/2 - (paddinglength/2 + 1) (jconvolutionalcodec.cpp:194) — AeroL's frame alignment relies on it. */
int jaero_viterbi_decode_continuous(jaero_viterbi *v, const uint8_t *soft, size_t n_soft,
                                    int interleaver_cols, uint8_t *bits_out, int32_t *n_valid);
int jaero_viterbi_decode_continuous_device(jaero_viterbi *v, const uint8_t *d_soft, size_t n_soft,
                                           int interleaver_cols, uint8_t *d_bits_out, int32_t *d_n_valid);
/* Decode_soft (one-shot, no overlap / padding): n_soft/2 bits out per channel. */
int jaero_viterbi_decode_block(jaero_viterbi *v, const uint8_t *soft, size_t n_soft, uint8_t *bits_out);
int jaero_viterbi_reset(jaero_viterbi *v);   /* SetCode(): clears the overlap of every channel */
int jaero_viterbi_sync(jaero_viterbi *v);
int64_t jaero_viterbi_launch_count(const jaero_viterbi *v);

/* ---- P-channel frame layer (600 / 1200 / 10500 bps, continuous): soft bits -> CRC-checked signal units ----
 * Replaces AeroL::processDemodulatedSoftBits -> AeroL::Decode(bits,true) (JAERO/aerol.cpp:2077-2090,1124-2039,
 * non-burst branch), AeroL::updateDCD (:1109-1122) and the DataCarrierDetect -> DCDstatSlot feedback
 * (JAERO/mainwindow.cpp:234-237). */
typedef struct jaero_pchannel jaero_pchannel;
int jaero_pchannel_create(int n_channels, double fb, int device_ordinal, jaero_pchannel **out);
void jaero_pchannel_destroy(jaero_pchannel *p);
/* Consume everything the batch's demodulators emitted since the last call (device-resident, no host hop),
 * run framing + de-interleave + Viterbi + descramble + CRC, and write each channel's DCD back into the batch. */
int jaero_pchannel_process_batch(jaero_pchannel *p, jaero_batch *b);
/* Same for soft bits supplied by the host: soft[ch*cap + k], counts[ch] (drop-in for processDemodulatedSoftBits). */
int jaero_pchannel_process_softbits(jaero_pchannel *p, const int16_t *soft, size_t cap_per_channel, const int32_t *counts);
/* AeroL::updateDCD: call once per second of signal (the reference's 1 s QTimer). b may be NULL. */
int jaero_pchannel_tick(jaero_pchannel *p, jaero_batch *b);
/* AeroL::SignalStatusSlot(false) -> AeroL::LostSignal() (JAERO/aerol.h:917-931): cntr = 1e9, DCD countdown = 0, DCD = false and
 * DataCarrierDetect(false) to the demodulator (b may be NULL: frame layer only). channel -1 = every channel. */
int jaero_pchannel_lost_signal(jaero_pchannel *p, jaero_batch *b, int channel);
/* writeData with the AeroL attached the way JAERO/mainwindow.cpp:198-237,432,508 wires the objects (HOST pcm): the stream is cut
 * in front of every coarse-estimator trigger sample and the frame layer runs at each cut, so FreqOffsetEstimateSlot reads the DCD
 * that results from exactly the soft bits emitted before that sample, and a SignalStatus(false) reaches LostSignal before any
 * later soft bit. Exact for OQPSK (DCD is only read in that slot); for MSK the timing-loop gain (mskdemodulator.cpp:387-405)
 * switches at the next cut, at most one estimator epoch (bbnfft/4 samples) after the reference's emit-granular switch.
 * Turns jaero_batch_wire_signal_status on for the batch. */
int jaero_pchannel_write_batch(jaero_pchannel *p, jaero_batch *b, const int16_t *pcm, size_t n_samples, size_t channel_stride);
/* Limits of one process call: a channel may hand over up to one full soft-bit ring (max(4096, 2*fb+64) values, i.e. 2 s of
 * signal at 10500 bps, 3.4 / 6.8 s at 1200 / 600 bps); more than that, or more signal units than jaero_pchannel_su_capacity()
 * left unread, raises the overflow flag: the next read_sus returns JAERO_E_OVERFLOW and the affected frames are incomplete. */
int jaero_pchannel_su_capacity(const jaero_pchannel *p);   /* SUs a channel can hold between two reads */
/* Drain decoded signal units: out[(ch*cap + k)*16 + 0..11] = SU bytes, [12] = CRC ok, [13] = index in frame,
 * [14..15] = frame number (LE). counts[ch] = SUs written. HOST pointers. */
int jaero_pchannel_read_sus(jaero_pchannel *p, uint8_t *out, size_t cap_per_channel, int32_t *counts);
/* Drop the queued signal units without copying them (device-side consumers / benchmarks). Asynchronous. */
int jaero_pchannel_discard_sus(jaero_pchannel *p);
/* dcd[ch], su_total[ch], su_ok[ch] (any may be NULL) */
int jaero_pchannel_get_stats(jaero_pchannel *p, int32_t *dcd, int64_t *su_total, int64_t *su_ok);
int64_t jaero_pchannel_launch_count(const jaero_pchannel *p);

/* ---- burst MSK demodulator (600 / 1200 bps R/T-channel bursts) ----
 * Replaces BurstMskDemodulator (JAERO/burstmskdemodulator.h:49-215): ctor + setSettings (burstmskdemodulator.cpp:11-323),
 * writeData (:371-754), DCDstatSlot (:757), and its processDemodulatedSoftBits / SignalStatus / EbNoMeasurmentSignal
 * signals. Soft-bit streams carry the reference's -1 "start of burst" marker. */
typedef struct jaero_burst jaero_burst;
typedef struct jaero_burst_status {
    double mixer2_freq, mixer2_wtptr, center_freq, st_freq, st_wtptr, agc, mse, ebno, vol_gain, rotator_freq;
    double n_sig_true, n_sig_false;   /* SignalStatus(true/false) emits */
    double cntr, startstop;
    double last_burst_ebno;           /* value of the most recent EbNoMeasurmentSignal */
    double n_ebno_emits;
} jaero_burst_status;
/* settings->kind is ignored; fb 600 or 1200, Fs 48000; freq_center / lockingbw / signalthreshold as BurstMskDemodulator::Settings */
int jaero_burst_msk_create(const jaero_settings *settings, int n_channels, int device_ordinal, jaero_burst **out);
/* Burst OQPSK demodulator (10500 bps C-channel / T-channel bursts): replaces BurstOqpskDemodulator
 * (JAERO/burstoqpskdemodulator.h), ctor + setSettings (burstoqpskdemodulator.cpp:4-277), writeData (:315-737) and its
 * processDemodulatedSoftBits / SignalStatus / EbNoMeasurmentSignal signals. fb 10500, Fs 48000; settings->sql as setSQL(). */
int jaero_burst_oqpsk_create(const jaero_settings *settings, int n_channels, int device_ordinal, jaero_burst **out);
void jaero_burst_destroy(jaero_burst *b);
int jaero_burst_write(jaero_burst *b, const int16_t *pcm, size_t n_samples, size_t channel_stride);          /* HOST pcm */
int jaero_burst_write_device(jaero_burst *b, const int16_t *d_pcm, size_t n_samples, size_t channel_stride);
int jaero_burst_read_softbits(jaero_burst *b, int16_t *out, size_t cap_per_channel, int32_t *counts);
int jaero_burst_set_dcd(jaero_burst *b, int channel, int dcd);
int jaero_burst_set_afc(jaero_burst *b, int state);                       /* setAFC (the constructors start with AFC on) */
int jaero_burst_set_sql(jaero_burst *b, int state);
int jaero_burst_get_status_all(jaero_burst *b, jaero_burst_status *out);
int jaero_burst_sync(jaero_burst *b);
int64_t jaero_burst_launch_count(const jaero_burst *b);

/* ---- R/T burst channel layer (SURVEY.md section 8(f)2) ----
 * Replaces the burst branch of AeroL::Decode (JAERO/aerol.cpp:1124-1350, :1985-2031: unique-word detection with the
 * start-of-burst timing gates, sync / time-out handling), AeroL::updateDCD (:1109-1122) and RTChannelDeleaveFECScram
 * (JAERO/aerol.h:554-895: trial de-interleave + Decode_soft at every candidate packet length, descrambling, CRC-16
 * decisions, byte packing). Input: the soft-bit stream a burst demodulator emits (values 0..255, -1 = start of burst).
 * Output records are JAERO_RT_RECORD bytes: int32 type (1 = R packet, 2 = T packet), int32 number of SUs (T), int32
 * payload length, int32 index of the packet's first bit, then the payload (R: 19 bytes; T: 6-byte header + 12 per SU). */
#define JAERO_RT_RECORD 400
typedef struct jaero_rt jaero_rt;
int jaero_rt_create(double fb, int n_channels, int device_ordinal, jaero_rt **out);     /* fb 600 / 1200 (MSK) or 10500 (OQPSK) */
void jaero_rt_destroy(jaero_rt *r);
/* host soft bits: soft[ch * cap + i], counts[ch] values per channel (AeroL::processDemodulatedSoftBits) */
int jaero_rt_process_softbits(jaero_rt *r, const int16_t *soft, size_t cap_per_channel, const int32_t *counts);
/* Opt-in vector semantics: AeroL::Decode returns in the middle of a soft-bit vector when the burst time-out fires
 * (JAERO/aerol.cpp:2018-2027) and the rest of that vector is lost. With it on, jaero_rt_process_burst drops the rest of the
 * demodulator's emit (12 / 32 values, +1 with the start marker) and jaero_rt_process_softbits treats each call as one vector.
 * Off (default): nothing is dropped. */
int jaero_rt_set_vector_mode(jaero_rt *r, int enabled);
/* consume (and drain) the soft bits a burst demodulator batch has produced, entirely on the device */
int jaero_rt_process_burst(jaero_rt *r, jaero_burst *b);
int jaero_rt_tick(jaero_rt *r);                                                          /* the 1 s updateDCD timer */
int jaero_rt_read_packets(jaero_rt *r, uint8_t *out, int cap_packets_per_channel, int32_t *counts);
int jaero_rt_get_stats(jaero_rt *r, int32_t *n_trial_decodes, int32_t *n_bad_packets, int32_t *dcd);   /* any may be NULL */
int64_t jaero_rt_launch_count(const jaero_rt *r);

/* ---- C-channel (8400 bps) frame layer (SURVEY.md section 8(f)3) ----
 * Replaces AeroL::DecodeC (JAERO/aerol.cpp:2187-2500): dual unique-word detector with I/Q ambiguity correction
 * (:848-896), 16 x (64 x 4) de-interleave, PuncturedCode::depunture_soft_block(...,4) (:2505-2518), Decode_Continuous,
 * delay line, scrambler, the three sub-band signal units per frame with CRC-16 + DCD countdown, the 25 x 12-byte voice
 * payload (what Voicesignal carries to the vocoder). Output records are JAERO_C_RECORD bytes: 3 x {12 SU bytes, crc_ok,
 * 3 pad}, 300 voice bytes, int32 frame number. */
#define JAERO_C_RECORD 352
typedef struct jaero_cchannel jaero_cchannel;
int jaero_cchannel_create(int n_channels, int device_ordinal, jaero_cchannel **out);
void jaero_cchannel_destroy(jaero_cchannel *c);
int jaero_cchannel_process_batch(jaero_cchannel *c, jaero_batch *b);      /* consume (and drain) an 8400 bps batch's soft bits on the device; DCD fed back */
int jaero_cchannel_process_softbits(jaero_cchannel *c, const int16_t *soft, size_t cap_per_channel, const int32_t *counts);
int jaero_cchannel_tick(jaero_cchannel *c, jaero_batch *b);               /* the 1 s updateDCD timer; b may be NULL */
int jaero_cchannel_lost_signal(jaero_cchannel *c, jaero_batch *b, int channel);   /* AeroL::LostSignal, as jaero_pchannel_lost_signal */
int jaero_cchannel_write_batch(jaero_cchannel *c, jaero_batch *b, const int16_t *pcm, size_t n_samples, size_t channel_stride);   /* as jaero_pchannel_write_batch */
int jaero_cchannel_read_frames(jaero_cchannel *c, uint8_t *out, int cap_frames_per_channel, int32_t *counts);
int jaero_cchannel_get_stats(jaero_cchannel *c, int32_t *dcd, int64_t *su_total, int64_t *su_ok);   /* any may be NULL */
int64_t jaero_cchannel_launch_count(const jaero_cchannel *c);

/* ---- ingest router (SURVEY.md section 8(f)4, host side) ----
 * The reference's many-channel feed is one ZMQ PUB topic per channel, each message three frames
 * [topic][uint32 sample rate][int16 PCM] (JAERO/zmq_audioreceiver.cpp:37-87; the subscription is the first 5 bytes of the
 * topic, :46) delivered to dataReceived(audio, sampleRate). The router takes the frames as the transport delivers them (no
 * libzmq dependency), files the PCM under the matching channel and feeds whole batches to jaero_batch_write. */
typedef struct jaero_ingest jaero_ingest;
int jaero_ingest_create(int n_channels, const char *const *topics, uint32_t sample_rate, size_t capacity_samples, jaero_ingest **out);
void jaero_ingest_destroy(jaero_ingest *g);
/* returns the channel index (>= 0) or a negative error. JAERO_E_OVERFLOW: the channel's buffer cannot take the whole message;
 * NOTHING of it was filed - flush the batch (jaero_ingest_flush) and hand the same message over again. */
int jaero_ingest_message(jaero_ingest *g, const void *topic, size_t topic_len, const void *rate, size_t rate_len, const void *pcm, size_t pcm_bytes);
size_t jaero_ingest_available(const jaero_ingest *g);                  /* samples every channel has */
int jaero_ingest_flush(jaero_ingest *g, jaero_batch *b, size_t n_samples);

/* ---- ISU / SSU reassembly and ACARS block parsing (SURVEY.md section 8(f)4, host side) ----
 * One handle per channel. Replaces RISUData::update (JAERO/aerol.cpp:27-112), ISUData::update (:151-214),
 * ParserISU::parse (:340-487) and ACARSDefragmenter (:221-329), fed the way AeroL::Decode feeds them (:1357-1399 R
 * packets, :1497-1513 T packets, :1900-1925 P-channel signal units). Pure host code, no device. The aircraft-database
 * look-up of ParserISU::acarslookupresult (:493-520) is not part of this library; only its removal of the leading dots of
 * the registration is applied. Input signal units must be CRC-valid (the device layers report crc_ok per unit). */
#define JAERO_REASM_ACARS 0      /* record kinds */
#define JAERO_REASM_ERROR 1      /* text = the reference's Errorsignal string */
#define JAERO_REASM_COMPLETE 1   /* push return bits: an ISU completed */
#define JAERO_REASM_MISSING 2    /* a subsequent signal unit had no open sequence */
#define JAERO_REASM_PARSED 4     /* the completed ISU was accepted by the parser */
#define JAERO_ACARS_NONACARS 1   /* flags: user data is not an ACARS block, text = its bytes in hex */
#define JAERO_ACARS_DOWNLINK 2
#define JAERO_ACARS_VALID 4
#define JAERO_ACARS_HASTEXT 8
#define JAERO_ACARS_MORE 16
typedef struct jaero_acars_record {
    int32_t kind;
    uint32_t aes_id;                 /* ISUItem: AESID, GESID, QNO, REFNO, SEQNO, NOOCTLESTINLASTSSU */
    uint8_t ges_id, qno, refno, seqno, last_octets;
    uint8_t mode, tak, block_id;     /* ACARSItem: MODE, TAK, BI */
    uint8_t label[2], label_len;     /* LABEL */
    uint8_t reg[7], reg_len;         /* PLANEREG */
    uint8_t flags;                   /* JAERO_ACARS_* */
    uint32_t userdata_len;           /* bytes of ISU user data the record was parsed from */
    uint32_t text_len;               /* bytes of message text (or error text) */
} jaero_acars_record;
typedef struct jaero_reasm jaero_reasm;
int jaero_reasm_create(jaero_reasm **out);
void jaero_reasm_destroy(jaero_reasm *h);
int jaero_reasm_reset(jaero_reasm *h);                                      /* AeroL::setSettings (:992-993) */
int jaero_reasm_short_frame(jaero_reasm *h);                                /* the short-frame reset (:1997) */
/* one P- or T-channel signal unit (first 10 of its 12 bytes are used); returns JAERO_REASM_* bits or a negative error */
int jaero_reasm_push_su(jaero_reasm *h, const uint8_t *su, int downlink);
/* one R-channel packet (first 17 of its 19 bytes are used) */
int jaero_reasm_push_r(jaero_reasm *h, const uint8_t *info, int downlink);
/* one T-channel packet as jaero_rt_read_packets returns it: 6-byte header + n_sus x 12 bytes */
int jaero_reasm_push_t_packet(jaero_reasm *h, const uint8_t *info, int n_sus);
int jaero_reasm_pending(const jaero_reasm *h);
/* pops the oldest record; returns the text length, -1 when there is none, -2 when cap < rec->text_len (nothing popped) */
long jaero_reasm_pop(jaero_reasm *h, jaero_acars_record *rec, char *text, size_t cap);
int jaero_reasm_get_stats(const jaero_reasm *h, uint64_t *isus, uint64_t *messages, uint64_t *errors, uint64_t *missing);   /* any may be NULL */

/* ---- device channelizer: one wideband complex IQ stream -> per-channel real audio rows for the demodulator batches ----
 * The reference has no channelizer (it takes audio from a sound card or ZMQ), so this definition is the contract.
 * x[n] counted from the handle's first write at input_rate (cs16: I,Q as they are; cu8: x = ((I-127.5) + j(Q-127.5)) * 256).
 * Rate change: L/M = output_rate / input_rate in lowest terms, accepted when 1 <= L <= 64 and M >= 2L. L is the smallest of
 * 1..64 for which r*L (r = input_rate / output_rate) lies within 1e-9 * r*L of an integer M; L = 1 is an integer ratio D = M.
 * Phases are uint32 fractions of a cycle: inc_c = llround(offset_c / input_rate * 2^32) mod 2^32, phi_c(n) = inc_c * n
 * mod 2^32, inc_a = llround(audio_hz / output_rate * 2^32), psi(m) = inc_a * m mod 2^32.
 * h[0..T-1] is the Kaiser low-pass prototype jaero_chan_taps returns, designed at L * input_rate and scaled to sum L (unity
 * DC gain in each of the L polyphase branches); h[j] = 0 for j >= T, Tp = ceil(T/L) taps per branch. Output m of channel c
 * sits at input time mM/L: n_m = floor(mM/L), p_m = mM mod L,
 *   a_c[m]   = sum_{k<Tp} h[kL + p_m] x[n_m - k] exp(-2 pi j phi_c(n_m - k) / 2^32)              (x[n<0] = 0)
 *   out_c[m] = saturate_int16(round_half_even(gain * Re{a_c[m] exp(2 pi j psi(m) / 2^32)}))
 * i.e. mix channel c to 0 Hz, resample by L/M (zero-stuff by L, low-pass at L*input_rate, keep every M-th sample), move it to
 * audio_hz, take the real part: the audio a batch with freq_center = audio_hz and Fs = output_rate expects. With L = 1,
 * n_m = mD and the sum runs over h[k] x[mD-k]. Filter: f_p = passband_hz/2, f_s = min(2 audio_hz, output_rate - 2 audio_hz)
 * - f_p (nearest alias / real-part fold into the passband), A = 60 dB, beta = 0.1102 (A - 8.7), T from Kaiser's estimate at
 * L * input_rate made odd (Tp <= 8191), cutoff (f_p + f_s)/2. */
#define JAERO_IQ_CS16 0
#define JAERO_IQ_CU8 1
#define JAERO_CHAN_MAX_TAPS 8191     /* per polyphase branch */
#define JAERO_CHAN_MAX_PHASES 64     /* largest L */
typedef struct jaero_chan_settings {
    int iq_format;                   /* JAERO_IQ_* */
    int reserved;
    double input_rate, output_rate;  /* Hz; output_rate / input_rate = L/M, L <= 64, M >= 2L */
    double audio_hz;                 /* where each channel's centre lands in the audio (= the batch's freq_center) */
    double passband_hz;              /* two-sided width kept within 0.05 dB */
    double gain;
} jaero_chan_settings;
typedef struct jaero_chan jaero_chan;
/* host only, no device: returns T (or a negative error), writes min(T, cap) taps of the prototype (sum L); taps may be NULL */
int jaero_chan_taps(const jaero_chan_settings *s, double *taps, int cap);
/* host only, no device: validates the settings as jaero_chan_taps does and returns the rate change L/M (either may be NULL) */
int jaero_chan_ratio(const jaero_chan_settings *s, int *L, int *M);
/* n_channels channels at offset_hz[c] from the IQ centre. Settings and offsets are validated before any device is touched. */
int jaero_chan_create(const jaero_chan_settings *s, int n_channels, const double *offset_hz, int device_ordinal, jaero_chan **out);
void jaero_chan_destroy(jaero_chan *c);
int jaero_chan_write(jaero_chan *c, const void *iq, size_t n_iq);           /* HOST iq, n_iq complex samples */
int jaero_chan_write_device(jaero_chan *c, const void *d_iq, size_t n_iq);  /* device iq; several handles may read the same buffer */
/* The audio produced by the most recent write (every output m with n_m inside the input so far), valid until the next write:
 * d_pcm[ch * channel_stride + i], i < n_samples; 16-byte aligned base, stride a multiple of 8 (jaero_batch_write_device takes
 * it as is). Ordered on the handle's stream. */
int jaero_chan_output_device(jaero_chan *c, const int16_t **d_pcm, size_t *n_samples, size_t *channel_stride);
/* copies the same rows to HOST out[ch * cap_per_channel + i]; *n_samples = samples per channel */
int jaero_chan_read(jaero_chan *c, int16_t *out, size_t cap_per_channel, size_t *n_samples);
int jaero_chan_set_stream(jaero_chan *c, void *cuda_stream);                /* as jaero_batch_set_stream */
int jaero_chan_sync(jaero_chan *c);
int64_t jaero_chan_launch_count(const jaero_chan *c);

#ifdef __cplusplus
}
#endif
#endif
