// Device lifecycle shared by the handles of the C ABI: opening a device, a create that fails part-way, the allocations a
// handle owns, grow-on-demand staging buffers and the stream link between a frame layer and a demodulator batch.
#pragma once
#include "common.cuh"
#include "../../include/jaero_b200.h"
#include <new>
#include <string>
#include <vector>

namespace jb {

// Select `device`, or fail with "<who>: no such CUDA device" (also when no CUDA device exists at all).
int open_device(int device, const char *who);

// The allocations a handle owns: zeroed device memory, device copies of host tables and pinned host memory, all freed
// together by free_all() when the handle is destroyed.
struct HandleAllocs {
    std::vector<void *> dev, host;
    template <class T> int zeroed(T **p, size_t count, cudaStream_t s)
    {
        JB_CUDA(cudaMalloc((void **)p, count * sizeof(T)));
        dev.push_back((void *)*p);
        JB_CUDA(cudaMemsetAsync(*p, 0, count * sizeof(T), s));
        return 0;
    }
    // src is copied before the call returns (pageable source), so it may go out of scope afterwards
    template <class T, class S> int upload(T **p, const std::vector<S> &src, cudaStream_t s)
    {
        static_assert(sizeof(T) == sizeof(S), "element layouts differ");
        JB_CUDA(cudaMalloc((void **)p, src.size() * sizeof(T)));
        dev.push_back((void *)*p);
        JB_CUDA(cudaMemcpyAsync(*p, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, s));
        return 0;
    }
    template <class T> int pinned(T **p, size_t count)
    {
        JB_CUDA(cudaMallocHost((void **)p, count * sizeof(T)));
        host.push_back((void *)*p);
        return 0;
    }
    void free_all()
    {
        for (void *q : dev) cudaFree(q);
        for (void *q : host) cudaFreeHost(q);
        dev.clear(); host.clear();
    }
};

// A device buffer that grows on demand. Growing waits for the work queued on `s`, which may still read the old buffer;
// a call that does not grow it costs nothing.
template <class T> struct GrowBuffer {
    T *ptr = nullptr;
    size_t cap = 0;             // elements
    int reserve(size_t count, cudaStream_t s)
    {
        if (count <= cap) return 0;
        JB_CUDA(cudaStreamSynchronize(s));
        release();
        JB_CUDA(cudaMalloc((void **)&ptr, count * sizeof(T)));
        cap = count;
        return 0;
    }
    void release() { cudaFree(ptr); ptr = nullptr; cap = 0; }
};

// Host soft bits of *_process_softbits, staged on the device: [C][cap] values and C counts.
struct SoftStage {
    GrowBuffer<int16_t> soft;
    GrowBuffer<int> counts;
    int upload(const int16_t *h_soft, size_t C, size_t cap, const int32_t *h_counts, cudaStream_t s)
    {
        if (soft.reserve(C * cap, s) || counts.reserve(C, s)) return JAERO_E_CUDA;
        JB_CUDA(cudaMemcpyAsync(soft.ptr, h_soft, C * cap * sizeof(int16_t), cudaMemcpyHostToDevice, s));
        JB_CUDA(cudaMemcpyAsync(counts.ptr, h_counts, C * sizeof(int), cudaMemcpyHostToDevice, s));
        return 0;
    }
    void release() { soft.release(); counts.release(); }
};

// Stream ordering between a frame layer's own stream and a demodulator batch's stream (which the layer never keeps: the
// batch may be destroyed first). Work launched on a batch's stream is followed by ev_batch, which the own stream waits
// for; work on the own stream sets own_dirty, and the next call that uses a batch's stream orders that stream behind ev_own.
struct StreamLink {
    cudaEvent_t ev_batch = 0, ev_own = 0;
    bool own_dirty = false;
    int create()
    {
        JB_CUDA(cudaEventCreateWithFlags(&ev_batch, cudaEventDisableTiming));
        JB_CUDA(cudaEventCreateWithFlags(&ev_own, cudaEventDisableTiming));
        return 0;
    }
    // a call is about to launch on the batch's stream `bs`: order it behind whatever the layer queued on `own`
    int enter(cudaStream_t own, cudaStream_t bs)
    {
        if (own_dirty) { JB_CUDA(cudaEventRecord(ev_own, own)); JB_CUDA(cudaStreamWaitEvent(bs, ev_own, 0)); own_dirty = false; }
        return 0;
    }
    // ... and `own` behind what was just launched on `bs`
    int leave(cudaStream_t own, cudaStream_t bs)
    {
        JB_CUDA(cudaEventRecord(ev_batch, bs)); JB_CUDA(cudaStreamWaitEvent(own, ev_batch, 0));
        return 0;
    }
    void destroy()
    {
        if (ev_batch) cudaEventDestroy(ev_batch);
        if (ev_own) cudaEventDestroy(ev_own);
    }
};

// The create preamble of a handle type T with members `int device` and `cudaStream_t stream`: select the device, make a
// value-initialised T with its own non-blocking stream. Until release(), leaving scope hands the partly built handle to its
// destroy function, so every early return of a create cleans up.
template <class T> struct NewHandle {
    T *h = nullptr;
    void (*destroy)(T *);
    explicit NewHandle(void (*d)(T *)) : destroy(d) {}
    ~NewHandle() { if (h) destroy(h); }
    NewHandle(const NewHandle &) = delete;
    NewHandle &operator=(const NewHandle &) = delete;
    int open(int device, const char *who)
    {
        int r = open_device(device, who);
        if (r) return r;
        h = new (std::nothrow) T();
        if (!h) { set_error("out of host memory"); return JAERO_E_ARG; }
        h->device = device;
        JB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        return JAERO_OK;
    }
    T *release() { T *t = h; h = nullptr; return t; }
};

} // namespace jb
