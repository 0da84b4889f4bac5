// runtime.cu -- device / memory / stream / event plumbing and the doubly mapped device ring.
//
// The ring replaces gr::cuda_buffer (reference runtime/lib/cudabuffer.cu:17-183), which
// emulates a circular buffer with a 2x allocation plus 1-3 cudaMemcpyAsync mirror copies and
// a cudaStreamSynchronize on every post_write.  Here one physical allocation is mapped twice
// back to back with the CUDA virtual memory management API -- the device analogue of the
// reference's host vmcirc buffer (runtime/lib/vmcircbuf_mmap_shm_open.cpp:92-121) -- so
// wrap-around windows are linearly addressable with zero extra traffic.
#include <cuda.h>

#include <mutex>

#include "common.cuh"

namespace b200 {

std::atomic<int64_t> g_launches{ 0 };

char* err_buf()
{
    static thread_local char buf[512] = { 0 };
    return buf;
}

int set_err(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(err_buf(), 512, fmt, ap);
    va_end(ap);
    return code;
}

int sm_count()
{
    // per-device, process-wide cache.  (Round 1 cached per THREAD and asked cudaGetDeviceProperties, which takes
    // 5-10 ms: every new scheduler thread paid that inside its first work() call -- most of a 10 ms flowgraph run.)
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
        return 148;
    int n = cache[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            return 148;
        cache[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

tmap_encode_fn tmap_encode_tiled()
{
    static tmap_encode_fn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (tmap_encode_fn)p;
    }();
    return fn;
}

// ---- driver entry points resolved through the runtime (no link-time libcuda dependency,
// so the library still loads on a machine without a driver) ------------------------------
struct drv_api {
    CUresult (*MemGetAllocationGranularity)(size_t*, const CUmemAllocationProp*,
                                            CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*MemAddressReserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*MemAddressFree)(CUdeviceptr, size_t) = nullptr;
    CUresult (*MemCreate)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*,
                          unsigned long long) = nullptr;
    CUresult (*MemRelease)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*MemMap)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle,
                       unsigned long long) = nullptr;
    CUresult (*MemUnmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*MemSetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*GetErrorString)(CUresult, const char**) = nullptr;
    bool ok = false;
};

static drv_api& drv()
{
    static drv_api api;
    static std::once_flag once;
    std::call_once(once, [] {
        auto get = [](const char* name, void** fn) {
            cudaDriverEntryPointQueryResult q;
            return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) == cudaSuccess &&
                   q == cudaDriverEntryPointSuccess && *fn;
        };
        bool ok = true;
        ok &= get("cuMemGetAllocationGranularity", (void**)&api.MemGetAllocationGranularity);
        ok &= get("cuMemAddressReserve", (void**)&api.MemAddressReserve);
        ok &= get("cuMemAddressFree", (void**)&api.MemAddressFree);
        ok &= get("cuMemCreate", (void**)&api.MemCreate);
        ok &= get("cuMemRelease", (void**)&api.MemRelease);
        ok &= get("cuMemMap", (void**)&api.MemMap);
        ok &= get("cuMemUnmap", (void**)&api.MemUnmap);
        ok &= get("cuMemSetAccess", (void**)&api.MemSetAccess);
        ok &= get("cuGetErrorString", (void**)&api.GetErrorString);
        api.ok = ok;
    });
    return api;
}

static const char* drv_err(CUresult r)
{
    const char* s = nullptr;
    if (drv().GetErrorString && drv().GetErrorString(r, &s) == CUDA_SUCCESS && s)
        return s;
    return "unknown driver error";
}

} // namespace b200

using namespace b200;

struct b200_ring {
    CUdeviceptr base = 0;
    size_t size = 0;
    CUmemGenericAllocationHandle handle = 0;
    int device = 0;
    bool mapped_lo = false, mapped_hi = false, have_handle = false;
};

extern "C" {

int b200_version(void) { return 101; }
const char* b200_last_error(void) { return err_buf(); }

int b200_device_count(int* count)
{
    if (!count)
        return set_err(B200_ERR_ARG, "count is null");
    B200_CUDA(cudaGetDeviceCount(count));
    return B200_OK;
}
int b200_set_device(int device)
{
    B200_CUDA(cudaSetDevice(device));
    return B200_OK;
}
int b200_get_device(int* device)
{
    if (!device)
        return set_err(B200_ERR_ARG, "device is null");
    B200_CUDA(cudaGetDevice(device));
    return B200_OK;
}
int b200_device_sm_count(int* sms)
{
    if (!sms)
        return set_err(B200_ERR_ARG, "sms is null");
    int dev = 0;
    B200_CUDA(cudaGetDevice(&dev));
    B200_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return B200_OK;
}
int b200_device_synchronize(void)
{
    B200_CUDA(cudaDeviceSynchronize());
    return B200_OK;
}
int64_t b200_launch_count(void) { return g_launches.load(); }

int b200_malloc(void** dptr, size_t bytes)
{
    if (!dptr)
        return set_err(B200_ERR_ARG, "dptr is null");
    B200_CUDA(cudaMalloc(dptr, bytes ? bytes : 1));
    return B200_OK;
}
int b200_free(void* dptr)
{
    B200_CUDA(cudaFree(dptr));
    return B200_OK;
}
int b200_host_alloc(void** hptr, size_t bytes)
{
    if (!hptr)
        return set_err(B200_ERR_ARG, "hptr is null");
    B200_CUDA(cudaHostAlloc(hptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return B200_OK;
}
int b200_host_free(void* hptr)
{
    B200_CUDA(cudaFreeHost(hptr));
    return B200_OK;
}
int b200_host_register(void* hptr, size_t bytes)
{
    B200_CUDA(cudaHostRegister(hptr, bytes, cudaHostRegisterDefault));
    return B200_OK;
}
int b200_host_unregister(void* hptr)
{
    B200_CUDA(cudaHostUnregister(hptr));
    return B200_OK;
}
int b200_memcpy_h2d(void* dst, const void* src, size_t bytes, b200_stream_t s)
{
    B200_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, cs(s)));
    return B200_OK;
}
int b200_memcpy_d2h(void* dst, const void* src, size_t bytes, b200_stream_t s)
{
    B200_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, cs(s)));
    return B200_OK;
}
int b200_memcpy_d2d(void* dst, const void* src, size_t bytes, b200_stream_t s)
{
    B200_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, cs(s)));
    return B200_OK;
}
int b200_memset(void* dst, int value, size_t bytes, b200_stream_t s)
{
    B200_CUDA(cudaMemsetAsync(dst, value, bytes, cs(s)));
    return B200_OK;
}
int b200_stream_create(b200_stream_t* s)
{
    if (!s)
        return set_err(B200_ERR_ARG, "s is null");
    cudaStream_t st;
    B200_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    *s = reinterpret_cast<b200_stream_t>(st);
    return B200_OK;
}
int b200_stream_destroy(b200_stream_t s)
{
    B200_CUDA(cudaStreamDestroy(cs(s)));
    return B200_OK;
}
int b200_stream_synchronize(b200_stream_t s)
{
    B200_CUDA(cudaStreamSynchronize(cs(s)));
    return B200_OK;
}
int b200_stream_wait_event(b200_stream_t s, b200_event_t e)
{
    B200_CUDA(cudaStreamWaitEvent(cs(s), reinterpret_cast<cudaEvent_t>(e), 0));
    return B200_OK;
}
int b200_event_create(b200_event_t* e, int timing)
{
    if (!e)
        return set_err(B200_ERR_ARG, "e is null");
    cudaEvent_t ev;
    B200_CUDA(cudaEventCreateWithFlags(&ev, timing ? cudaEventDefault : cudaEventDisableTiming));
    *e = reinterpret_cast<b200_event_t>(ev);
    return B200_OK;
}
int b200_event_destroy(b200_event_t e)
{
    B200_CUDA(cudaEventDestroy(reinterpret_cast<cudaEvent_t>(e)));
    return B200_OK;
}
int b200_event_record(b200_event_t e, b200_stream_t s)
{
    B200_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(e), cs(s)));
    return B200_OK;
}
int b200_event_synchronize(b200_event_t e)
{
    B200_CUDA(cudaEventSynchronize(reinterpret_cast<cudaEvent_t>(e)));
    return B200_OK;
}
int b200_event_query(b200_event_t e)
{
    cudaError_t r = cudaEventQuery(reinterpret_cast<cudaEvent_t>(e));
    if (r == cudaSuccess)
        return 0;
    if (r == cudaErrorNotReady)
        return 1;
    return set_err(B200_ERR_CUDA, "cudaEventQuery -> %s", cudaGetErrorString(r));
}
int b200_event_elapsed_ms(b200_event_t start, b200_event_t stop, float* ms)
{
    if (!ms)
        return set_err(B200_ERR_ARG, "ms is null");
    B200_CUDA(cudaEventElapsedTime(ms, reinterpret_cast<cudaEvent_t>(start),
                                   reinterpret_cast<cudaEvent_t>(stop)));
    return B200_OK;
}

// ---- peer memory: another GPU's buffer addressed directly by this GPU's kernels (NVLink loads),
// the multi-GPU halo path (SURVEY.md 8e): no exchange step, no copy, nothing on the critical path.
int b200_enable_peer_access(int peer_device)
{
    int dev = 0, can = 0;
    B200_CUDA(cudaGetDevice(&dev));
    if (peer_device == dev)
        return B200_OK;
    B200_CUDA(cudaDeviceCanAccessPeer(&can, dev, peer_device));
    if (!can)
        return set_err(B200_ERR_UNSUPPORTED, "device %d cannot access device %d", dev, peer_device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return B200_OK;
    }
    B200_CUDA(e);
    return B200_OK;
}

// makes the device a stream lives on the calling thread's current device (kernel launches need it; copies and
// event operations do not).  Host blocks call it at the top of work(): one flowgraph process can then drive
// several GPUs, one scheduler thread per block as in the reference (thread_wrapper.cpp:21).
int b200_stream_activate(b200_stream_t s)
{
    int dev = -1, cur = -1;
    B200_CUDA(cudaStreamGetDevice(cs(s), &dev));
    B200_CUDA(cudaGetDevice(&cur));
    if (dev != cur)
        B200_CUDA(cudaSetDevice(dev));
    return B200_OK;
}

int b200_ipc_export(const void* dptr, b200_ipc_handle* out)
{
    if (!dptr || !out)
        return set_err(B200_ERR_ARG, "ipc_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    memset(out, 0, sizeof(*out));
    void* base = nullptr;
    size_t size = 0;
    {
        static CUresult (*get_range)(CUdeviceptr*, size_t*, CUdeviceptr) = [] {
            void* fn = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q) != cudaSuccess ||
                q != cudaDriverEntryPointSuccess)
                fn = nullptr;
            return (CUresult(*)(CUdeviceptr*, size_t*, CUdeviceptr))fn;
        }();
        if (!get_range)
            return set_err(B200_ERR_CUDA, "ipc_export: cuMemGetAddressRange unavailable");
        CUdeviceptr b = 0;
        CUresult r = get_range(&b, &size, (CUdeviceptr)dptr);
        if (r != CUDA_SUCCESS)
            return set_err(B200_ERR_CUDA, "ipc_export: cuMemGetAddressRange -> %s", drv_err(r));
        base = (void*)b;
    }
    cudaIpcMemHandle_t h;
    B200_CUDA(cudaIpcGetMemHandle(&h, base));
    memcpy(out->bytes, &h, 64);
    out->offset = (uint64_t)((const char*)dptr - (const char*)base);
    out->size = size;
    int dev = 0;
    B200_CUDA(cudaGetDevice(&dev));
    out->device = dev;
    return B200_OK;
}

int b200_ipc_import(const b200_ipc_handle* h, void** dptr)
{
    if (!h || !dptr)
        return set_err(B200_ERR_ARG, "ipc_import: null argument");
    cudaIpcMemHandle_t mh;
    memcpy(&mh, h->bytes, 64);
    void* base = nullptr;
    B200_CUDA(cudaIpcOpenMemHandle(&base, mh, cudaIpcMemLazyEnablePeerAccess));
    *dptr = (char*)base + h->offset;
    return B200_OK;
}

int b200_ipc_close(const b200_ipc_handle* h, void* dptr)
{
    if (!h || !dptr)
        return set_err(B200_ERR_ARG, "ipc_close: null argument");
    B200_CUDA(cudaIpcCloseMemHandle((char*)dptr - h->offset));
    return B200_OK;
}

// ------------------------------------------------------------------------------- ring
static int ring_prop(CUmemAllocationProp* prop, int* dev_out)
{
    int dev = 0;
    B200_CUDA(cudaGetDevice(&dev));
    B200_CUDA(cudaFree(0)); // make sure the primary context exists
    memset(prop, 0, sizeof(*prop));
    prop->type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop->location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop->location.id = dev;
    if (dev_out)
        *dev_out = dev;
    return B200_OK;
}

size_t b200_ring_granularity(void)
{
    CUmemAllocationProp prop;
    if (ring_prop(&prop, nullptr) != B200_OK || !drv().ok)
        return 0;
    size_t g = 0;
    if (drv().MemGetAllocationGranularity(&g, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) !=
        CUDA_SUCCESS)
        return 0;
    return g;
}

int b200_ring_destroy(b200_ring* r)
{
    if (!r)
        return B200_OK;
    drv_api& d = drv();
    if (r->mapped_lo)
        d.MemUnmap(r->base, r->size);
    if (r->mapped_hi)
        d.MemUnmap(r->base + r->size, r->size);
    if (r->have_handle)
        d.MemRelease(r->handle);
    if (r->base)
        d.MemAddressFree(r->base, 2 * r->size);
    delete r;
    return B200_OK;
}

int b200_ring_create(size_t min_bytes, b200_ring** ring)
{
    if (!ring || min_bytes == 0)
        return set_err(B200_ERR_ARG, "ring_create: null out pointer or zero size");
    *ring = nullptr;
    drv_api& d = drv();
    CUmemAllocationProp prop;
    int dev = 0;
    int rc = ring_prop(&prop, &dev);
    if (rc != B200_OK)
        return rc;
    if (!d.ok)
        return set_err(B200_ERR_CUDA, "ring_create: CUDA VMM driver entry points unavailable");
    size_t gran = 0;
    CUresult cr = d.MemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED);
    if (cr != CUDA_SUCCESS || gran == 0)
        return set_err(B200_ERR_CUDA, "cuMemGetAllocationGranularity -> %s", drv_err(cr));
    size_t size = (min_bytes + gran - 1) / gran * gran;

    b200_ring* r = new b200_ring();
    r->size = size;
    r->device = dev;
#define RING_DRV(call)                                                              \
    do {                                                                            \
        CUresult c__ = (call);                                                      \
        if (c__ != CUDA_SUCCESS) {                                                  \
            b200_ring_destroy(r);                                                   \
            return set_err(c__ == CUDA_ERROR_OUT_OF_MEMORY ? B200_ERR_NOMEM         \
                                                           : B200_ERR_CUDA,         \
                           "ring_create: %s -> %s", #call, drv_err(c__));           \
        }                                                                           \
    } while (0)
    RING_DRV(d.MemAddressReserve(&r->base, 2 * size, gran, 0, 0));
    RING_DRV(d.MemCreate(&r->handle, size, &prop, 0));
    r->have_handle = true;
    RING_DRV(d.MemMap(r->base, size, 0, r->handle, 0));
    r->mapped_lo = true;
    RING_DRV(d.MemMap(r->base + size, size, 0, r->handle, 0));
    r->mapped_hi = true;
    CUmemAccessDesc acc;
    memset(&acc, 0, sizeof(acc));
    acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    acc.location.id = dev;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    RING_DRV(d.MemSetAccess(r->base, 2 * size, &acc, 1));
#undef RING_DRV
    *ring = r;
    return B200_OK;
}

// lets kernels and copy engines of `peer_device` address this ring (VMM allocations are private to the
// device they were granted to until cuMemSetAccess says otherwise)
int b200_ring_enable_peer(b200_ring* r, int peer_device)
{
    if (!r)
        return set_err(B200_ERR_ARG, "ring_enable_peer: null ring");
    if (peer_device == r->device)
        return B200_OK;
    CUmemAccessDesc acc;
    memset(&acc, 0, sizeof(acc));
    acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    acc.location.id = peer_device;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    CUresult c = drv().MemSetAccess(r->base, 2 * r->size, &acc, 1);
    if (c != CUDA_SUCCESS)
        return set_err(B200_ERR_CUDA, "ring_enable_peer: cuMemSetAccess -> %s", drv_err(c));
    return B200_OK;
}

void* b200_ring_base(const b200_ring* r) { return r ? reinterpret_cast<void*>(r->base) : nullptr; }
size_t b200_ring_size(const b200_ring* r) { return r ? r->size : 0; }

} // extern "C"

// ---- FP32 FMA peak probe (denominator for the FP32-bound FIR roofline; SURVEY.md 8d says the
// driver's MEASURED_PEAKS.json has no FP32 figure and the build must measure it) -------------
namespace b200 {
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float a, float b)
{
    float r[16];
#pragma unroll
    for (int i = 0; i < 16; i++)
        r[i] = (float)(threadIdx.x + i);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 16; u++)
#pragma unroll
            for (int i = 0; i < 16; i++)
                r[i] = fmaf(r[i], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++)
        s += r[i];
    if (s == 12345.678f)
        out[0] = s;
}
} // namespace b200

extern "C" int b200_measure_fp32_tflops(int iters, float* tflops, float* ms_out)
{
    if (iters < 1 || !tflops)
        return set_err(B200_ERR_ARG, "measure_fp32_tflops: bad argument");
    float* d = nullptr;
    B200_CUDA(cudaMalloc(&d, 4));
    cudaEvent_t e0, e1;
    B200_CUDA(cudaEventCreate(&e0));
    B200_CUDA(cudaEventCreate(&e1));
    const int blocks = sm_count() * 8;
    B200_LAUNCH(fp32_peak_kernel, blocks, 256, 0, 0, d, 16, 1.0001f, 0.5f); // warm-up
    B200_CUDA(cudaEventRecord(e0, 0));
    B200_LAUNCH(fp32_peak_kernel, blocks, 256, 0, 0, d, iters, 1.0001f, 0.5f);
    B200_CUDA(cudaEventRecord(e1, 0));
    B200_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    double flops = 2.0 * 256.0 * (double)blocks * 256.0 * (double)iters;
    *tflops = (float)(flops / (ms * 1e-3) / 1e12);
    if (ms_out)
        *ms_out = ms;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    return B200_OK;
}

namespace b200 {
__global__ void __launch_bounds__(256) fp32x2_peak_kernel(float* out, int iters, float a, float b)
{
    float2 r[8];
#pragma unroll
    for (int i = 0; i < 8; i++)
        r[i] = make_float2((float)(threadIdx.x + i), (float)(threadIdx.x - i));
    const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 16; u++)
#pragma unroll
            for (int i = 0; i < 8; i++)
                r[i] = __ffma2_rn(r[i], a2, b2);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++)
        s += r[i].x + r[i].y;
    if (s == 12345.678f)
        out[0] = s;
}
} // namespace b200

extern "C" int b200_measure_fp32x2_tflops(int iters, float* tflops, float* ms_out)
{
    if (iters < 1 || !tflops)
        return set_err(B200_ERR_ARG, "measure_fp32x2_tflops: bad argument");
    float* d = nullptr;
    B200_CUDA(cudaMalloc(&d, 4));
    cudaEvent_t e0, e1;
    B200_CUDA(cudaEventCreate(&e0));
    B200_CUDA(cudaEventCreate(&e1));
    const int blocks = sm_count() * 8;
    B200_LAUNCH(fp32x2_peak_kernel, blocks, 256, 0, 0, d, 16, 1.0001f, 0.5f);
    B200_CUDA(cudaEventRecord(e0, 0));
    B200_LAUNCH(fp32x2_peak_kernel, blocks, 256, 0, 0, d, iters, 1.0001f, 0.5f);
    B200_CUDA(cudaEventRecord(e1, 0));
    B200_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    double flops = 2.0 * 256.0 * (double)blocks * 256.0 * (double)iters;
    *tflops = (float)(flops / (ms * 1e-3) / 1e12);
    if (ms_out)
        *ms_out = ms;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    return B200_OK;
}
