// Handle structs of the C ABI that more than one handle family reaches into: the demodulator batch (frame layers and the
// ingest router feed it and drain its soft-bit ring) and the burst demodulator (the R/T layer drains its ring).
#pragma once
#include "handle.cuh"
#include "demod.cuh"
#include "prefilter.cuh"
#include "burst.cuh"
#include <utility>

namespace jb {

// The estimator-trigger schedule of a batch (oqpskdemodulator.cpp:410-431), the same for every channel: bb is the
// reference's bbcycbuff_ptr, cc its coarseCounter and phys the matching slot of the device ring (bb_len slots).
struct TriggerSchedule {
    int bb = 0, cc = 0, phys = 0;
    // A(i) for one sample: the ring write advances the counters; true when the sample triggers a coarse estimate, which
    // restarts coarseCounter
    bool step(const DemodParams &p)
    {
        const int N = p.bbnfft, trig_every = p.cpu_reduce ? N : N / 4;
        bool trigger = false;
        if (cc >= p.Fs || !p.cpu_reduce) {
            bb++; if (bb >= N) bb = 0;
            phys++; if (phys >= p.bb_len) phys = 0;
            if (bb % trig_every == 0) trigger = true;
        }
        if (trigger) cc = 0;                                       // :426
        cc++;                                                      // :431
        return trigger;
    }
};

// Copy the soft-bit rings of C channels to host rows of `cap` values through the pinned stage [C][soft_cap]; cnt / ovf are
// the host copies of the per-channel counts and overflow flags. JAERO_E_OVERFLOW when a ring overflowed or holds more than
// cap values; the rings are not reset here.
int read_soft_rows(const int *cnt, const int *ovf, int C, const int16_t *d_soft, int soft_cap, int16_t *h_stage, int16_t *out,
                   size_t cap, int32_t *counts, cudaStream_t s);

} // namespace jb

struct jaero_batch {
    int device;
    cudaStream_t stream, own_stream;    // stream: the caller's (jaero_batch_set_stream) or own_stream
    jb::HandleAllocs allocs;
    jaero_settings set;
    jb::DemodParams p;
    jb::CfePlan cfe;
    long long samples;                  // samples fully processed
    jb::TriggerSchedule trig;           // lock-step counters mirrored on the host
    jb::GrowBuffer<int16_t> stage;      // host input, or re-pitched unaligned device input
    // 8400 bps pre-filter (K6)
    bool pre_on; jb::PreParams pre; jb::FirStream fir; int fir_fill; long long fir_blocks; jb::GrowBuffer<double2> x;
    int16_t *h_soft_stage;              // pinned
    int *h_ints; double *h_dbls; long long *h_soft_total;   // pinned mirrors of I / D / soft_total
    long long launches;
    bool profiling;
    // asynchronous coarse estimator (see jaero_batch_write_device)
    bool async_cfe; cudaStream_t cfe_stream; cudaEvent_t ev_seg_done, ev_cfe_done[2]; int cfe_count;
    // host-input pipelining (jaero_batch_write): the H2D copy is cut into column slices on a copy stream; a segment only
    // waits for the slices it reads
    cudaStream_t copy_stream; cudaEvent_t ev_slice[8], ev_stage_free; int n_slices, slice_len, next_slice;
    bool use_pipe;              // 10500 bps: warp-specialised segment kernel (JAERO_OQPSK_PIPE=0 selects the single-warp one, for A/B profiling)
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_seg, ev_cfe;
    double prof_samples;
    int trace_state;            // JAERO_PIPE_TRACE: 0 = armed, 1 = done
    // seating of the channels in the pipelined 10500 bps kernel (regroup)
    int *d_chan_of; double *d_keys, *h_keys; double *d_ring_scratch;
    std::vector<int> slot_of;   // [cpad] seat of channel c
    long long epochs, next_regroup; int regroup_every; long long regroups;
};

struct jaero_burst {
    int device; cudaStream_t stream;
    jb::HandleAllocs allocs;
    jb::BurstParams p; jb::HilbertStream hil;
    long long samples; int hil_fill; long long hil_blocks;
    jb::GrowBuffer<int16_t> stage;
    double2 *tw32k, *wa, *wb; int *d_ev_list; int ev_round;
    int *h_ints; double *h_dbls; int16_t *h_soft;
    std::vector<int> h_ev;
    long long launches;
};

namespace jb {
// move the not-yet-emitted soft bits of every channel to the front of its ring, after the frame layer or a host read
// consumed the rest (launched on the owner's stream)
int batch_soft_reset(const jaero_batch *b, cudaStream_t s);
int burst_soft_reset(const jaero_burst *b, cudaStream_t s);
} // namespace jb
