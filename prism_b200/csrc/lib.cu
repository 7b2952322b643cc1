// lib.cu -- library-level entry points of libprism_b200.so
#include "common.cuh"

std::atomic<long long> g_pb_launches{0};

int pb_sm_count()
{
    static std::atomic<int> cached[64];
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return n;
    const int c = cached[dev].load(std::memory_order_relaxed);
    if (c > 0) return c;
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) n = v;
    cached[dev].store(n, std::memory_order_relaxed);
    return n;
}

namespace {
// device timeline mark: the GPU's nanosecond clock at the point of the stream (or graph branch) it was enqueued on
__global__ void stamp_kernel(unsigned long long *dst)
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    *dst = t;
}
}  // namespace

extern "C" {

int pb_stamp_time(unsigned long long *dst, void *stream)
{
    if (!dst) return PB_E_ARG;
    PB_LAUNCH(stamp_kernel, 1, 1, 0, stream, dst);
    return PB_OK;
}

int pb_abi_version(void) { return PB_ABI_VERSION; }

long long pb_launch_count(void) { return g_pb_launches.load(std::memory_order_relaxed); }

// ---- thin stream / event / copy wrappers: the per-iteration host path of the fused ingest issues its staging copy
// and its cross-stream ordering through these (one ctypes call each) instead of framework context managers.
int pb_event_create(void **event)
{
    if (!event) return PB_E_ARG;
    cudaEvent_t e;
    cudaError_t rc = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (rc != cudaSuccess) return (int)rc;
    *event = (void *)e;
    return PB_OK;
}
int pb_event_destroy(void *event) { return event ? (int)cudaEventDestroy((cudaEvent_t)event) : PB_OK; }
int pb_event_record(void *event, void *stream) { return (int)cudaEventRecord((cudaEvent_t)event, (cudaStream_t)stream); }
int pb_event_synchronize(void *event) { return (int)cudaEventSynchronize((cudaEvent_t)event); }
int pb_stream_wait_event(void *stream, void *event) { return (int)cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)event, 0); }
int pb_copy_h2d_async(void *dst, const void *src, long long bytes, void *stream)
{
    if (!dst || !src || bytes < 0) return PB_E_ARG;
    return (int)cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream);
}
int pb_copy_d2h_async(void *dst, const void *src, long long bytes, void *stream)
{
    if (!dst || !src || bytes < 0) return PB_E_ARG;
    return (int)cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
}

// The fused ingest's per-iteration submission as ONE host call: on copy_stream wait for after_event (NULL: nothing to wait
// for), copy the pinned block to the device, record copied_event; main_stream then waits for copied_event.
int pb_staged_copy_submit(void *copy_stream, void *after_event, void *dst, const void *src, long long bytes,
                          void *copied_event, void *main_stream)
{
    if (!dst || !src || bytes < 0 || !copied_event) return PB_E_ARG;
    cudaStream_t cs = (cudaStream_t)copy_stream;
    cudaError_t e = cudaSuccess;
    if (after_event) e = cudaStreamWaitEvent(cs, (cudaEvent_t)after_event, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, cs);
    if (e == cudaSuccess) e = cudaEventRecord((cudaEvent_t)copied_event, cs);
    if (e == cudaSuccess) e = cudaStreamWaitEvent((cudaStream_t)main_stream, (cudaEvent_t)copied_event, 0);
    return (int)e;
}

int pb_copy_d2d_async(void *dst, const void *src, long long bytes, void *stream)
{
    if (!dst || !src || bytes < 0) return PB_E_ARG;
    return (int)cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
}

const char *pb_error_string(int code)
{
    switch (code) {
        case PB_OK: return "ok";
        case PB_E_ARG: return "invalid argument";
        case PB_E_CAPACITY: return "capacity must be a power of two in [32, 2^30] with size <= capacity";
        case PB_E_UNSUPPORTED: return "unsupported option";
        case PB_E_POOL: return "aux observation pool exhausted";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown error";
}

}  // extern "C"
