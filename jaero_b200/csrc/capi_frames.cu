// C ABI of the frame layers: P-channel (jaero_pchannel_*), C-channel (jaero_cchannel_*) and burst R/T (jaero_rt_*). The P- and
// C-channel layers drain a demodulator batch's soft-bit ring on the batch's stream and keep their own stream ordered with it;
// the code they share is written once below, parameterised by the layer's kernel calls.
#include "capi_internal.cuh"
#include "host_design.h"
#include "pchannel.cuh"
#include "cchannel.cuh"
#include "rtchannel.cuh"
#include <cstring>

using namespace jb;

struct jaero_pchannel {
    int device; cudaStream_t stream;
    HandleAllocs allocs;
    StreamLink link;
    SoftStage stage;
    PChanParams pp;
    uint8_t *vit_overlap; int *vit_overlap_len, *vit_renorm, *vit_valid;
    PChanState *h_state; uint8_t *h_su;
    long long launches;
};

struct jaero_cchannel {
    int device; cudaStream_t stream;
    HandleAllocs allocs;
    StreamLink link;
    SoftStage stage;
    CChanParams cp;
    uint8_t *vit_overlap; int *vit_overlap_len, *vit_renorm, *vit_valid;
    CChanState *h_state; uint8_t *h_out;
    long long launches;
};

struct jaero_rt {
    int device; cudaStream_t stream;
    HandleAllocs allocs;
    SoftStage stage;
    RtParams rp;
    RtState *h_state; uint8_t *h_out;
    long long launches;
    int vector_mode;
};

namespace {

// ---- P- and C-channel layers (L = jaero_pchannel or jaero_cchannel)
// create: event pair of the stream link and the per-channel state of the layer's continuous Viterbi decoder
template <class L> int frame_layer_init(L *l, size_t C)
{
    if (l->link.create()) return JAERO_E_CUDA;
    HandleAllocs &A = l->allocs;
    if (A.zeroed(&l->vit_overlap, C * 64, l->stream) || A.zeroed(&l->vit_overlap_len, C, l->stream) ||
        A.zeroed(&l->vit_renorm, C, l->stream) || A.zeroed(&l->vit_valid, C, l->stream)) return JAERO_E_CUDA;
    return JAERO_OK;
}
// the layer queues work on batch streams, so destroy waits for the whole device
template <class L> void frame_layer_destroy(L *l)
{
    if (!l) return;
    cudaSetDevice(l->device);
    cudaDeviceSynchronize();
    l->allocs.free_all(); l->stage.release(); l->link.destroy();
    if (l->stream) cudaStreamDestroy(l->stream);
    delete l;
}
// process_batch: `process(dp)` drains the batch's soft-bit ring on the batch's stream, ordered after the demodulator segments;
// the ring is reset behind it
template <class L, class F> int frame_process_batch(L *l, jaero_batch *b, F process)
{
    JB_CUDA(cudaSetDevice(l->device));
    if (l->link.enter(l->stream, b->stream)) return JAERO_E_CUDA;
    if (process(b->p) || batch_soft_reset(b, b->stream)) return JAERO_E_CUDA;
    l->launches++;
    return l->link.leave(l->stream, b->stream) ? JAERO_E_CUDA : JAERO_OK;
}
// tick / lost_signal: `launch(demod_dcd, stream)` runs on the batch's stream with its DCD row when a batch is given (b may be
// NULL: frame layer only, on the layer's own stream)
template <class L, class F> int frame_call(L *l, jaero_batch *b, F launch)
{
    JB_CUDA(cudaSetDevice(l->device));
    if (b) { if (l->link.enter(l->stream, b->stream)) return JAERO_E_CUDA; } else l->link.own_dirty = true;
    if (launch(b ? b->p.I + (size_t)I_DCD * b->p.cpad : nullptr, b ? b->stream : l->stream)) return JAERO_E_CUDA;
    l->launches++;
    return (b && l->link.leave(l->stream, b->stream)) ? JAERO_E_CUDA : JAERO_OK;
}
// Length of the piece of a write that ends in front of the next coarse-estimator trigger sample (the only points where the OQPSK
// demodulator reads DCD and where SignalStatus is emitted): the batch's trigger schedule, stepped on a copy.
size_t piece_before_next_trigger(const jaero_batch *b, size_t n)
{
    TriggerSchedule t = b->trig;
    for (size_t i = 0; i < n; i++)
        if (t.step(b->p) && i > 0) return i;                       // a trigger on the first sample opens this piece
    return n;
}
// writeData with the AeroL attached the way JAERO/mainwindow.cpp:198-237,432,508 wires them: the stream is cut in front of
// every estimator trigger sample and the frame layer runs at each cut, so that the DCD the demodulator reads in
// FreqOffsetEstimateSlot, and the LostSignal that follows a SignalStatus(false), see exactly the soft bits emitted before
// that sample (exact for OQPSK, whose only reads of DCD are in that slot; for MSK the timing-loop gain switches at the next
// cut, at most one estimator epoch after the reference's emit-granular switch). HOST pcm.
template <class L> int frame_write_batch(L *l, jaero_batch *b, const int16_t *pcm, size_t n, size_t stride, int (*process)(L *, jaero_batch *))
{
    b->p.wire_sigstat = 1;
    size_t done = 0;
    while (done < n) {
        const size_t k = piece_before_next_trigger(b, n - done);   // >= 1: up to, not including, the next trigger sample
        int rc = jaero_batch_write(b, pcm + done, k, stride);
        if (rc) return rc;
        rc = process(l, b);
        if (rc) return rc;
        done += k;
    }
    return JAERO_OK;
}

// ---- all frame layers
template <class S> int pull_state(S *h_state, const S *d_state, size_t C, cudaStream_t s)
{
    JB_CUDA(cudaMemcpyAsync(h_state, d_state, C * sizeof(S), cudaMemcpyDeviceToHost, s));
    JB_CUDA(cudaStreamSynchronize(s));
    return 0;
}
// DCD and signal-unit counters of the P- and C-channel layers
template <class S> int su_stats(S *h_state, const S *d_state, size_t C, cudaStream_t s, int32_t *dcd, int64_t *su_total, int64_t *su_ok)
{
    if (pull_state(h_state, d_state, C, s)) return JAERO_E_CUDA;
    for (size_t ch = 0; ch < C; ch++) {
        if (dcd) dcd[ch] = h_state[ch].datacd;
        if (su_total) su_total[ch] = h_state[ch].su_total;
        if (su_ok) su_ok[ch] = h_state[ch].su_ok;
    }
    return JAERO_OK;
}
// Copy the output records of C channels (a ring of `ring` records of `rec` bytes each, state[ch].out_count of them filled) to
// host rows of `cap` records. *overflow: a queue overflowed or held more than cap records.
template <class S> int read_records(S *h_state, const S *d_state, uint8_t *h_out, const uint8_t *d_out, size_t C, int ring, size_t rec,
                                    uint8_t *out, int cap, int32_t *counts, cudaStream_t s, bool *overflow)
{
    JB_CUDA(cudaMemcpyAsync(h_state, d_state, C * sizeof(S), cudaMemcpyDeviceToHost, s));
    JB_CUDA(cudaMemcpyAsync(h_out, d_out, C * ring * rec, cudaMemcpyDeviceToHost, s));
    JB_CUDA(cudaStreamSynchronize(s));
    *overflow = false;
    for (size_t ch = 0; ch < C; ch++) {
        const int n = h_state[ch].out_count;
        *overflow |= h_state[ch].overflow != 0 || n > cap;
        counts[ch] = n < cap ? n : cap;
        for (int k = 0; k < counts[ch]; k++) memcpy(out + (ch * cap + k) * rec, h_out + (ch * ring + k) * rec, rec);
    }
    return 0;
}

__global__ void pchan_su_reset_kernel(PChanParams pp)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch < pp.n_channels) { pp.state[ch].su_count = 0; pp.state[ch].queue_overflow = 0; }
}
} // namespace

extern "C" {

// ====================================================================== P-channel frame layer
int jaero_pchannel_create(int n_channels, double fb, int device, jaero_pchannel **out)
{
    PChanParams pp;
    const char *bad = out ? pchannel_plan(n_channels, fb, pp) : "jaero_pchannel_create: bad argument";
    if (bad) { set_error(bad); return JAERO_E_ARG; }
    NewHandle<jaero_pchannel> nh(jaero_pchannel_destroy);
    int r = nh.open(device, "jaero_pchannel_create"); if (r) return r;
    jaero_pchannel *p = nh.h;
    p->pp = pp;
    PChanParams &q = p->pp;
    HandleAllocs &A = p->allocs;
    const size_t C = n_channels;
    cudaStream_t st = p->stream;
    int rc = frame_layer_init(p, C);
    rc |= A.zeroed(&q.state, C, st);
    rc |= A.zeroed(&q.blocks, C * q.queue * q.block_len, st);
    rc |= A.zeroed(&q.decoded, C * q.queue * (q.block_len / 2), st);
    rc |= A.zeroed(&q.meta, C * q.queue, st);
    rc |= A.zeroed(&q.ready, C, st);
    rc |= A.zeroed(&q.dl2, C * q.dl2_len, st);
    rc |= A.zeroed(&q.infofield, C * q.info_cap, st);
    rc |= A.zeroed(&q.su_out, C * q.su_cap * 16, st);
    if (rc || pchan_set_scrambler(scrambler_sequence(5000).data()) || pchan_init(q, st)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(st));
    if (A.pinned(&p->h_state, C) || A.pinned(&p->h_su, C * q.su_cap * 16)) return JAERO_E_CUDA;
    *out = nh.release();
    return JAERO_OK;
}
void jaero_pchannel_destroy(jaero_pchannel *p) { frame_layer_destroy(p); }
int64_t jaero_pchannel_launch_count(const jaero_pchannel *p) { return p ? p->launches : 0; }
int jaero_pchannel_su_capacity(const jaero_pchannel *p) { return p ? p->pp.su_cap : 0; }

int jaero_pchannel_process_batch(jaero_pchannel *p, jaero_batch *b)
{
    if (!p || !b || p->pp.n_channels != b->p.n_channels || p->device != b->device) { set_error("jaero_pchannel_process_batch: batch mismatch"); return JAERO_E_ARG; }
    return frame_process_batch(p, b, [&](const DemodParams &dp) {
        return pchan_process(p->pp, dp.soft, dp.I + (size_t)I_SOFT_COUNT * dp.cpad, dp.soft_cap, dp.I + (size_t)I_DCD * dp.cpad, p->vit_overlap,
                             p->vit_overlap_len, p->vit_renorm, p->vit_valid, p->pp.queue, b->stream, &p->launches,
                             dp.I + (size_t)I_LOST_N * dp.cpad, dp.lost_pos, dp.cpad);
    });
}
int jaero_pchannel_process_softbits(jaero_pchannel *p, const int16_t *soft, size_t cap, const int32_t *counts)
{
    if (!p || !soft || !counts || cap == 0) { set_error("jaero_pchannel_process_softbits: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(p->device));
    p->link.own_dirty = true;
    if (p->stage.upload(soft, p->pp.n_channels, cap, counts, p->stream)) return JAERO_E_CUDA;
    if (pchan_process(p->pp, p->stage.soft.ptr, p->stage.counts.ptr, (int)cap, nullptr, p->vit_overlap, p->vit_overlap_len,
                      p->vit_renorm, p->vit_valid, p->pp.queue, p->stream, &p->launches)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(p->stream));
    return JAERO_OK;
}
int jaero_pchannel_tick(jaero_pchannel *p, jaero_batch *b)
{
    if (!p || (b && b->p.n_channels != p->pp.n_channels)) { set_error("jaero_pchannel_tick: bad argument"); return JAERO_E_ARG; }
    return frame_call(p, b, [&](int *dcd, cudaStream_t s) { return pchan_tick(p->pp, dcd, s); });
}
// AeroL::SignalStatusSlot(false) -> LostSignal() (aerol.h:920-931): cntr = 1e9, DCD countdown and DCD cleared at once, and
// DataCarrierDetect(false) reaches the demodulator (b may be NULL: frame layer only). channel -1 = every channel.
int jaero_pchannel_lost_signal(jaero_pchannel *p, jaero_batch *b, int channel)
{
    if (!p || channel >= p->pp.n_channels || (b && b->p.n_channels != p->pp.n_channels)) { set_error("jaero_pchannel_lost_signal: bad argument"); return JAERO_E_ARG; }
    return frame_call(p, b, [&](int *dcd, cudaStream_t s) { return pchan_lost(p->pp, channel, dcd, s); });
}
int jaero_pchannel_write_batch(jaero_pchannel *p, jaero_batch *b, const int16_t *pcm, size_t n, size_t stride)
{
    if (!p || !b || !pcm || p->pp.n_channels != b->p.n_channels || p->device != b->device) { set_error("jaero_pchannel_write_batch: bad argument"); return JAERO_E_ARG; }
    if (stride < n) { set_error("jaero_pchannel_write_batch: channel_stride < n_samples"); return JAERO_E_ARG; }
    return frame_write_batch(p, b, pcm, n, stride, jaero_pchannel_process_batch);
}
int jaero_pchannel_read_sus(jaero_pchannel *p, uint8_t *out, size_t cap, int32_t *counts)
{
    if (!p || !out || !counts) { set_error("jaero_pchannel_read_sus: null argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(p->device));
    const PChanParams &pp = p->pp;
    if (pull_state(p->h_state, pp.state, pp.n_channels, p->stream)) return JAERO_E_CUDA;   // p->stream is ordered behind every batch-stream call
    bool overflow = false; int maxc = 0;
    for (int ch = 0; ch < pp.n_channels; ch++) { maxc = std::max(maxc, p->h_state[ch].su_count); overflow |= p->h_state[ch].queue_overflow != 0 || (size_t)p->h_state[ch].su_count > cap; }
    if (overflow) { set_error("P-channel queue overflow: call process/read more often"); return JAERO_E_OVERFLOW; }
    if (maxc) { JB_CUDA(cudaMemcpyAsync(p->h_su, pp.su_out, (size_t)pp.n_channels * pp.su_cap * 16, cudaMemcpyDeviceToHost, p->stream)); JB_CUDA(cudaStreamSynchronize(p->stream)); }
    for (int ch = 0; ch < pp.n_channels; ch++) {
        counts[ch] = p->h_state[ch].su_count;
        if (counts[ch]) memcpy(out + (size_t)ch * cap * 16, p->h_su + (size_t)ch * pp.su_cap * 16, (size_t)counts[ch] * 16);
    }
    pchan_su_reset_kernel<<<(pp.n_channels + 127) / 128, 128, 0, p->stream>>>(pp);
    JB_CUDA(cudaGetLastError());
    p->link.own_dirty = true;
    return JAERO_OK;
}
int jaero_pchannel_discard_sus(jaero_pchannel *p)
{
    if (!p) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(p->device));
    pchan_su_reset_kernel<<<(p->pp.n_channels + 127) / 128, 128, 0, p->stream>>>(p->pp);
    JB_CUDA(cudaGetLastError());
    p->link.own_dirty = true;
    p->launches++;
    return JAERO_OK;
}
int jaero_pchannel_get_stats(jaero_pchannel *p, int32_t *dcd, int64_t *su_total, int64_t *su_ok)
{
    if (!p) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(p->device));
    return su_stats(p->h_state, p->pp.state, p->pp.n_channels, p->stream, dcd, su_total, su_ok);
}

// ====================================================================== R/T burst channel layer (§8(f)2)
int jaero_rt_create(double fb, int n_channels, int device, jaero_rt **out)
{
    RtParams rp;
    const char *bad = out ? rt_plan(fb, n_channels, rp) : "jaero_rt_create: bad argument";
    if (bad) { set_error(bad); return JAERO_E_ARG; }
    NewHandle<jaero_rt> nh(jaero_rt_destroy);
    int r = nh.open(device, "jaero_rt_create"); if (r) return r;
    jaero_rt *t = nh.h;
    t->rp = rp;
    RtParams &q = t->rp;
    HandleAllocs &A = t->allocs;
    const size_t C = n_channels;
    cudaStream_t st = t->stream;
    int rc = 0;
    rc |= A.zeroed(&q.state, C, st); rc |= A.zeroed(&q.slots, C * RT_SLOTS, st); rc |= A.zeroed(&q.blocks, C * RT_SLOTS * RT_BLOCK, st);
    rc |= A.zeroed(&q.out, C * RT_OUT * RT_OUT_BYTES, st);
    if (rc || rt_set_scrambler(scrambler_sequence(5000).data()) || rt_init(q, st)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(st));
    if (A.pinned(&t->h_state, C) || A.pinned(&t->h_out, C * RT_OUT * RT_OUT_BYTES)) return JAERO_E_CUDA;
    *out = nh.release();
    return JAERO_OK;
}
void jaero_rt_destroy(jaero_rt *r)
{
    if (!r) return;
    cudaSetDevice(r->device);
    cudaStreamSynchronize(r->stream);
    r->allocs.free_all(); r->stage.release();
    cudaStreamDestroy(r->stream);
    delete r;
}
int64_t jaero_rt_launch_count(const jaero_rt *r) { return r ? r->launches : 0; }

int jaero_rt_process_softbits(jaero_rt *r, const int16_t *soft, size_t cap, const int32_t *counts)
{
    if (!r || !soft || !counts || cap == 0) { set_error("jaero_rt_process_softbits: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(r->device));
    if (r->stage.upload(soft, r->rp.n_channels, cap, counts, r->stream)) return JAERO_E_CUDA;
    if (rt_process(r->rp, r->stage.soft.ptr, r->stage.counts.ptr, cap, r->stream, &r->launches, r->vector_mode ? -1 : 0)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(r->stream));
    return JAERO_OK;
}
int jaero_rt_process_burst(jaero_rt *r, jaero_burst *b)
{
    if (!r || !b || r->rp.n_channels != b->p.n_channels || r->device != b->device) { set_error("jaero_rt_process_burst: demodulator mismatch"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(r->device));
    const BurstParams &bp = b->p;
    JB_CUDA(cudaStreamSynchronize(r->stream));
    // on the demodulator's stream: ordered after its kernels; its soft ring is drained afterwards
    if (rt_process(r->rp, bp.soft, bp.BI + (size_t)BI_SOFT_COUNT * bp.cpad, (size_t)bp.soft_cap, b->stream, &r->launches,
                   r->vector_mode ? (bp.kind == 1 ? 32 : 12) : 0)) return JAERO_E_CUDA;   // emit sizes: burstoqpskdemodulator.cpp / burstmskdemodulator.cpp:735
    if (burst_soft_reset(b, b->stream)) return JAERO_E_CUDA;
    r->launches++;
    JB_CUDA(cudaStreamSynchronize(b->stream));
    return JAERO_OK;
}
// Opt-in: reproduce AeroL::Decode's return in the middle of a soft-bit vector when the burst time-out fires (aerol.cpp:2018-2027)
int jaero_rt_set_vector_mode(jaero_rt *r, int enabled)
{
    if (!r) { set_error("null handle"); return JAERO_E_ARG; }
    r->vector_mode = enabled ? 1 : 0;
    return JAERO_OK;
}
int jaero_rt_tick(jaero_rt *r)
{
    if (!r) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(r->device));
    if (rt_tick(r->rp, r->stream)) return JAERO_E_CUDA;
    r->launches++;
    return JAERO_OK;
}
int jaero_rt_read_packets(jaero_rt *r, uint8_t *out, int cap_packets, int32_t *counts)
{
    if (!r || !out || !counts || cap_packets <= 0) { set_error("jaero_rt_read_packets: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(r->device));
    bool overflow;
    if (read_records(r->h_state, r->rp.state, r->h_out, r->rp.out, r->rp.n_channels, RT_OUT, RT_OUT_BYTES, out, cap_packets, counts, r->stream, &overflow) ||
        rt_out_reset(r->rp, r->stream)) return JAERO_E_CUDA;
    r->launches++;
    if (overflow) { set_error("R/T packet queue overflow: read more often"); return JAERO_E_OVERFLOW; }
    return JAERO_OK;
}
int jaero_rt_get_stats(jaero_rt *r, int32_t *n_trials, int32_t *n_bad, int32_t *dcd)
{
    if (!r) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(r->device));
    const size_t C = r->rp.n_channels;
    if (pull_state(r->h_state, r->rp.state, C, r->stream)) return JAERO_E_CUDA;
    for (size_t ch = 0; ch < C; ch++) {
        if (n_trials) n_trials[ch] = r->h_state[ch].n_trials;
        if (n_bad) n_bad[ch] = r->h_state[ch].n_bad;
        if (dcd) dcd[ch] = r->h_state[ch].datacd;
    }
    return JAERO_OK;
}

// ====================================================================== C-channel (8400 bps) frame layer (§8(f)3)
int jaero_cchannel_create(int n_channels, int device, jaero_cchannel **out)
{
    if (!out || n_channels <= 0) { set_error("jaero_cchannel_create: bad argument"); return JAERO_E_ARG; }
    NewHandle<jaero_cchannel> nh(jaero_cchannel_destroy);
    int r = nh.open(device, "jaero_cchannel_create"); if (r) return r;
    jaero_cchannel *c = nh.h;
    CChanParams &cp = c->cp;
    cp.n_channels = n_channels; cp.dl2_len = 2714 - 6 + 1;                     // dl2.setLength(2714-6) (aerol.cpp:1037)
    HandleAllocs &A = c->allocs;
    const size_t C = n_channels;
    cudaStream_t st = c->stream;
    int rc = frame_layer_init(c, C);
    rc |= A.zeroed(&cp.state, C, st); rc |= A.zeroed(&cp.coded, C * CC_QUEUE * CC_CODED_PITCH, st); rc |= A.zeroed(&cp.decoded, C * CC_QUEUE * CC_DEC, st);
    rc |= A.zeroed(&cp.ready, C, st); rc |= A.zeroed(&cp.dl2, C * cp.dl2_len, st); rc |= A.zeroed(&cp.out, C * CC_OUT * CC_RECORD, st);
    if (rc || cchan_set_scrambler(scrambler_sequence(5000).data()) || cchan_init(cp, st)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(st));
    if (A.pinned(&c->h_state, C) || A.pinned(&c->h_out, C * CC_OUT * CC_RECORD)) return JAERO_E_CUDA;
    *out = nh.release();
    return JAERO_OK;
}
void jaero_cchannel_destroy(jaero_cchannel *c) { frame_layer_destroy(c); }
int64_t jaero_cchannel_launch_count(const jaero_cchannel *c) { return c ? c->launches : 0; }

int jaero_cchannel_process_batch(jaero_cchannel *c, jaero_batch *b)
{
    if (!c || !b || c->cp.n_channels != b->p.n_channels || c->device != b->device) { set_error("jaero_cchannel_process_batch: batch mismatch"); return JAERO_E_ARG; }
    return frame_process_batch(c, b, [&](const DemodParams &dp) {
        return cchan_process(c->cp, dp.soft, dp.I + (size_t)I_SOFT_COUNT * dp.cpad, (size_t)dp.soft_cap, dp.I + (size_t)I_DCD * dp.cpad, c->vit_overlap,
                             c->vit_overlap_len, c->vit_renorm, c->vit_valid, b->stream, &c->launches, dp.I + (size_t)I_LOST_N * dp.cpad, dp.lost_pos, dp.cpad);
    });
}
int jaero_cchannel_process_softbits(jaero_cchannel *c, const int16_t *soft, size_t cap, const int32_t *counts)
{
    if (!c || !soft || !counts || cap == 0) { set_error("jaero_cchannel_process_softbits: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    c->link.own_dirty = true;
    if (c->stage.upload(soft, c->cp.n_channels, cap, counts, c->stream)) return JAERO_E_CUDA;
    if (cchan_process(c->cp, c->stage.soft.ptr, c->stage.counts.ptr, cap, nullptr, c->vit_overlap, c->vit_overlap_len, c->vit_renorm, c->vit_valid,
                      c->stream, &c->launches)) return JAERO_E_CUDA;
    JB_CUDA(cudaStreamSynchronize(c->stream));
    return JAERO_OK;
}
int jaero_cchannel_tick(jaero_cchannel *c, jaero_batch *b)
{
    if (!c || (b && b->p.n_channels != c->cp.n_channels)) { set_error("jaero_cchannel_tick: bad argument"); return JAERO_E_ARG; }
    return frame_call(c, b, [&](int *dcd, cudaStream_t s) { return cchan_tick(c->cp, dcd, s); });
}
int jaero_cchannel_lost_signal(jaero_cchannel *c, jaero_batch *b, int channel)     // AeroL::LostSignal, see jaero_pchannel_lost_signal
{
    if (!c || channel >= c->cp.n_channels || (b && b->p.n_channels != c->cp.n_channels)) { set_error("jaero_cchannel_lost_signal: bad argument"); return JAERO_E_ARG; }
    return frame_call(c, b, [&](int *dcd, cudaStream_t s) { return cchan_lost(c->cp, channel, dcd, s); });
}
int jaero_cchannel_write_batch(jaero_cchannel *c, jaero_batch *b, const int16_t *pcm, size_t n, size_t stride)
{
    if (!c || !b || !pcm || c->cp.n_channels != b->p.n_channels || c->device != b->device) { set_error("jaero_cchannel_write_batch: bad argument"); return JAERO_E_ARG; }
    if (stride < n) { set_error("jaero_cchannel_write_batch: channel_stride < n_samples"); return JAERO_E_ARG; }
    return frame_write_batch(c, b, pcm, n, stride, jaero_cchannel_process_batch);
}
int jaero_cchannel_read_frames(jaero_cchannel *c, uint8_t *out, int cap_frames, int32_t *counts)
{
    if (!c || !out || !counts || cap_frames <= 0) { set_error("jaero_cchannel_read_frames: bad argument"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    bool overflow;
    if (read_records(c->h_state, c->cp.state, c->h_out, c->cp.out, c->cp.n_channels, CC_OUT, CC_RECORD, out, cap_frames, counts, c->stream, &overflow) ||
        cchan_out_reset(c->cp, c->stream)) return JAERO_E_CUDA;
    c->link.own_dirty = true;
    c->launches++;
    if (overflow) { set_error("C-channel frame queue overflow: read more often"); return JAERO_E_OVERFLOW; }
    return JAERO_OK;
}
int jaero_cchannel_get_stats(jaero_cchannel *c, int32_t *dcd, int64_t *su_total, int64_t *su_ok)
{
    if (!c) { set_error("null handle"); return JAERO_E_ARG; }
    JB_CUDA(cudaSetDevice(c->device));
    return su_stats(c->h_state, c->cp.state, c->cp.n_channels, c->stream, dcd, su_total, su_ok);
}

} // extern "C"
