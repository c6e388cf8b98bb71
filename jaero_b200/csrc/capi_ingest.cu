// C ABI of the ingest router (jaero_ingest_*): host-side filing of per-channel PCM messages for a demodulator batch.
#include "capi_internal.cuh"
#include <algorithm>
#include <cstring>

using namespace jb;

// The many-channel feed of the reference: one ZMQ PUB topic per channel, every message three frames
// [topic][uint32 sample rate][int16 PCM] (JAERO/zmq_audioreceiver.cpp:37-87, subscription = the first 5 bytes of the
// topic, :46), delivered to the demodulator's dataReceived(audio, sampleRate) slot (oqpskdemodulator.cpp:686-693).
// This router takes the three frames as the transport hands them over (no libzmq dependency), files the PCM under the
// channel whose topic matches and, once every channel has n samples, feeds them to a batch in one jaero_batch_write.
struct jaero_ingest {
    int n_channels; uint32_t rate; size_t cap;
    std::vector<std::string> topics;
    std::vector<int16_t> pcm;               // [n_channels][cap]
    std::vector<size_t> fill;
    long long dropped_bytes, messages;
};

extern "C" {

int jaero_ingest_create(int n_channels, const char *const *topics, uint32_t sample_rate, size_t capacity_samples, jaero_ingest **out)
{
    if (!out || !topics || n_channels <= 0 || capacity_samples == 0) { set_error("jaero_ingest_create: bad argument"); return JAERO_E_ARG; }
    jaero_ingest *g = new (std::nothrow) jaero_ingest();
    if (!g) { set_error("out of host memory"); return JAERO_E_ARG; }
    g->n_channels = n_channels; g->rate = sample_rate; g->cap = capacity_samples; g->dropped_bytes = 0; g->messages = 0;
    for (int c = 0; c < n_channels; c++) {
        if (!topics[c]) { delete g; set_error("jaero_ingest_create: null topic"); return JAERO_E_ARG; }
        g->topics.push_back(std::string(topics[c]).substr(0, 5));          // zmq_setsockopt(..., ZMQ_SUBSCRIBE, topic, 5)
    }
    g->pcm.assign((size_t)n_channels * capacity_samples, 0);
    g->fill.assign(n_channels, 0);
    *out = g;
    return JAERO_OK;
}
void jaero_ingest_destroy(jaero_ingest *g) { delete g; }

int jaero_ingest_message(jaero_ingest *g, const void *topic, size_t topic_len, const void *rate, size_t rate_len, const void *pcm, size_t pcm_bytes)
{
    if (!g || !topic || !rate || (!pcm && pcm_bytes)) { set_error("jaero_ingest_message: null argument"); return JAERO_E_ARG; }
    if (rate_len != 4) { set_error("jaero_ingest_message: the sample-rate frame must be 4 bytes"); return JAERO_E_ARG; }
    uint32_t r; memcpy(&r, rate, 4);                                           // memcpy(&sampleRate, rate, 4) (:70)
    int ch = -1;
    for (int c = 0; c < g->n_channels && ch < 0; c++) {
        const std::string &t = g->topics[c];
        if (topic_len >= t.size() && memcmp(topic, t.data(), t.size()) == 0) ch = c;   // prefix match, as a ZMQ subscription does
    }
    if (ch < 0) { set_error("jaero_ingest_message: no channel subscribes to this topic"); return JAERO_E_ARG; }
    if (r != g->rate) { set_error("jaero_ingest_message: sample rate differs from the batch's (the reference re-applies its settings; a batch is fixed-rate)"); return JAERO_E_STATE; }
    g->messages++;
    size_t n = pcm_bytes / 2;                                                   // writeData: len/2 int16 samples
    const size_t room = g->cap - g->fill[ch];
    // a full channel buffer refuses the whole message (nothing is filed, so the caller can flush and re-send): dropping
    // the tail silently would desynchronise this channel against the lock-step batch
    if (n > room) { g->dropped_bytes += (long long)n * 2; set_error("jaero_ingest_message: channel buffer full (flush the batch, then re-send this message)"); return JAERO_E_OVERFLOW; }
    memcpy(g->pcm.data() + (size_t)ch * g->cap + g->fill[ch], pcm, n * 2);
    g->fill[ch] += n;
    return ch;
}
size_t jaero_ingest_available(const jaero_ingest *g)
{
    if (!g) return 0;
    size_t m = g->cap;
    for (int c = 0; c < g->n_channels; c++) m = std::min(m, g->fill[c]);
    return m;
}
int jaero_ingest_flush(jaero_ingest *g, jaero_batch *b, size_t n)
{
    if (!g || !b || b->p.n_channels != g->n_channels) { set_error("jaero_ingest_flush: batch mismatch"); return JAERO_E_ARG; }
    if (n == 0) return JAERO_OK;
    if (n > jaero_ingest_available(g)) { set_error("jaero_ingest_flush: not every channel has that many samples"); return JAERO_E_STATE; }
    const int rc = jaero_batch_write(b, g->pcm.data(), n, g->cap);
    if (rc != JAERO_OK) return rc;
    JB_CUDA(cudaStreamSynchronize(b->stream));                                 // the pageable staging rows are reused below
    for (int c = 0; c < g->n_channels; c++) {
        int16_t *row = g->pcm.data() + (size_t)c * g->cap;
        memmove(row, row + n, (g->fill[c] - n) * 2);
        g->fill[c] -= n;
    }
    return JAERO_OK;
}

} // extern "C"
