// Host-side design of every handle: filter taps, delay weights, spectra, tables and the scalar kernel parameters a create
// call derives from its settings. Plain C++ (no CUDA runtime calls), so a CPU test can pin every value; the kernels depend
// on these values bit for bit, so the loop orders and expression forms are those of the reference's own code.
#pragma once
#include "common.cuh"
#include "demod.cuh"
#include "burst.cuh"
#include "prefilter.cuh"
#include "pchannel.cuh"
#include "rtchannel.cuh"
#include "../../include/jaero_b200.h"
#include <complex>
#include <cstdint>
#include <vector>

namespace jb {

typedef std::vector<std::complex<double>> cvec;

// RootRaisedCosine::design (JAERO/DSP.h:316-338): closed-form RRC taps, firsize forced odd.
std::vector<double> rrc_taps(double alpha, int firsize, double samplerate, double symbol_freq);
// Delay<T>::update (JAERO/DSP.h:357-374) at every position bp of its ceil(fd)+1 ring: w[bp] is the interpolation weight the
// reference derives from (buffptr - fractdelay). Returns whether the read position is "ceil(fd) samples ago" at every ring
// position, which the shift-register form of the kernels needs.
bool delay_weights(double fd, std::vector<double> &w);
// W_n^k = exp(-2 pi i k / n), k < n
cvec twiddles(int n);
// in-place radix-2 FFT (bit reversal, then butterflies) with the table of twiddles(x.size())
void fft_radix2(cvec &x, const cvec &tw);
// TrigLookUp (JAERO/DSP.cpp:19-20): the 19999-entry sine and cosine tables
void trig_tables(std::vector<double> &sn, std::vector<double> &cs);
// AeroLScrambler::pre_state (JAERO/aerol.h:397-419): the first n bits of the descrambling sequence
std::vector<uint8_t> scrambler_sequence(int n);
// CoarseFreqEstimate::setSettings (coarsefreqestimate.cpp:62-74): raised-cosine window of the 8400 bps estimator
std::vector<double> estimator_window(int nfft, int startbin);

// Everything jaero_batch_create derives from its settings before it touches a device. A non-null return is the
// message of an unsupported setting (JAERO_E_ARG).
struct BatchPlan {
    DemodParams p;          // scalar fields and taps; device pointers, bb_len and chan_of are left zero
    CfePlan cfe;            // scalar fields; group and clusters are left zero
    double st_freq;         // initial symbol-timing oscillator frequency
    cvec cfe_tw;            // estimator twiddles, nfft entries
    std::vector<double> cfe_window;   // 8400 bps only
    cvec pre_H, pre_tw;     // 8400 bps pre-filter: spectrum of the 2049-tap RRC and W_4096^k
};
const char *batch_plan(const jaero_settings *s, int n_channels, BatchPlan &plan);

// Everything burst_create derives from its settings (kind 0 = MSK, 1 = OQPSK).
struct BurstPlan {
    BurstParams p;          // scalar fields and taps
    HilbertStream hil;      // K, nfft, L
    double freq_center;     // clamped initial mixer frequency
    std::vector<double> w_btd1, w_btdiff, w_a1;   // Delay<> weight per ring position
    cvec hil_H, hil_tw, tw32k;                    // Hilbert spectrum, W_8192^k, W_32768^k
};
const char *burst_plan(const jaero_settings *s, int n_channels, int kind, BurstPlan &plan);

// Frame-layer sizing of jaero_pchannel_create and jaero_rt_create (scalar fields only).
const char *pchannel_plan(int n_channels, double fb, PChanParams &pp);
const char *rt_plan(double fb, int n_channels, RtParams &rp);

} // namespace jb
