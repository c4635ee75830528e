// Contexts, errors, kernel timing, and the NCCL binding behind the communicators of the one-process-per-GPU exchange.

#include <dlfcn.h>
#include <stdlib.h>

#include "host_state.h"

using namespace e2s;

namespace e2s {

// ---- NCCL, bound at run time (no link dependency: under Python the process already holds torch's libnccl.so.2, a
// stand-alone CLI gets the system one).  Only the five calls the inter-phase exchange needs; ABI as in nccl.h 2.x. ----
typedef struct { char internal[128]; } e2s_nccl_id;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(e2s_nccl_id*) = nullptr;
    int (*CommInitRank)(void**, int, e2s_nccl_id, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // already in the process (torch)?
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (h) {
            api.lib = h;
            api.GetUniqueId = reinterpret_cast<int (*)(e2s_nccl_id*)>(dlsym(h, "ncclGetUniqueId"));
            api.CommInitRank = reinterpret_cast<int (*)(void**, int, e2s_nccl_id, int)>(dlsym(h, "ncclCommInitRank"));
            api.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(h, "ncclAllGather"));
            api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
            api.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
            if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather || !api.CommDestroy) api.lib = nullptr;
        }
    }
    return api.lib ? &api : nullptr;
}
constexpr int NCCL_UINT64 = 5;  // ncclUint64 (nccl.h: ncclDataType_t)

thread_local std::string g_err;

int fail(e2s_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    g_err = msg;
    return code;
}
int cuda_fail(e2s_ctx* ctx, cudaError_t e, const char* what) {
    return fail(ctx, E2S_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// every rank's exchange row (cm->d_send) into cm->d_recv, on the context's stream
int all_gather_rows(e2s_ctx* c, e2s_comm* cm) {
    NcclApi* na = nccl_api();
    const int nr = na->AllGather(cm->d_send, cm->d_recv, XR_WORDS, NCCL_UINT64, cm->nccl, c->stream);
    if (nr != 0) return fail(c, E2S_ERR_CUDA, std::string("ncclAllGather: ") + (na->GetErrorString ? na->GetErrorString(nr) : "error"));
    return E2S_OK;
}

}  // namespace e2s

extern "C" {

int e2s_version(void) { return E2S_VERSION; }

const char* e2s_last_error(const e2s_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

int e2s_ctx_create(int device, e2s_ctx** out) {
    if (!out) return fail(nullptr, E2S_ERR_ARG, "e2s_ctx_create: out == NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, E2S_ERR_CUDA,
                    std::string("no CUDA device (this library has no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, E2S_ERR_ARG, "e2s_ctx_create: bad device index");
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, E2S_ERR_CUDA, "device is not sm_100 class: the kernels are built for sm_100a only");
    int sm_count = prop.multiProcessorCount;
    if (const char* e = getenv("E2S_SM_COUNT")) {  // test hook: size every grid for fewer SMs, so CTAs loop at small inputs
        char* end = nullptr;
        const long v = strtol(e, &end, 10);
        if (end == e || *end || v < 1 || v > prop.multiProcessorCount)
            return fail(nullptr, E2S_ERR_ARG, std::string("E2S_SM_COUNT=") + e + ": expected 1.." +
                                                  std::to_string(prop.multiProcessorCount) + " (the device's SM count)");
        sm_count = int(v);
    }
    CU(nullptr, cudaSetDevice(device));
    e2s_ctx* c = new e2s_ctx();
    c->device = device;
    c->sm_count = sm_count;
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return cuda_fail(nullptr, e, "cudaStreamCreate");
    }
    c->own_stream = true;
    *out = c;
    return E2S_OK;
}

void e2s_ctx_destroy(e2s_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->cached) e2s_shard_destroy(c->cached);
    if (c->reads_owned) {
        cudaFree(c->d_bases);
        cudaFree(c->d_off);
    }
    cudaFree(c->d_raw[0]);
    cudaFree(c->d_raw[1]);
    cudaFree(c->d_reads_flag);
    for (int i = 0; i < 2; ++i) {
        if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
        if (c->ev_soa_staged[i]) cudaEventDestroy(c->ev_soa_staged[i]);
        if (c->ev_soa_free[i]) cudaEventDestroy(c->ev_soa_free[i]);
        cudaFree(c->d_soa_stage[i]);
        if (c->ev_unpacked[i]) cudaEventDestroy(c->ev_unpacked[i]);
    }
    if (c->ev_start) cudaEventDestroy(c->ev_start);
    for (int i = 0; i < 4; ++i)
        if (c->ev_slot[i]) cudaEventDestroy(c->ev_slot[i]);
    if (c->pin_ring) cudaFreeHost(c->pin_ring);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int e2s_ctx_set_stream(e2s_ctx* c, void* s) {
    if (!c) return fail(nullptr, E2S_ERR_ARG, "ctx == NULL");
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    c->stream = static_cast<cudaStream_t>(s);
    c->own_stream = false;
    return E2S_OK;
}

int e2s_ctx_synchronize(e2s_ctx* c) {
    if (!c) return fail(nullptr, E2S_ERR_ARG, "ctx == NULL");
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    return E2S_OK;
}

uint64_t e2s_ctx_launch_count(const e2s_ctx* c) { return c ? c->launches : 0; }

int e2s_ctx_timing(e2s_ctx* c, int enable) {
    if (!c) return fail(nullptr, E2S_ERR_ARG, "ctx == NULL");
    c->timer.enabled = enable != 0;
    if (enable) {  // events for a few dozen steps up front: none is created inside a timed region
        CU(c, cudaSetDevice(c->device));
        while (c->timer.pool.size() < 512) {
            cudaEvent_t e;
            CU(c, cudaEventCreate(&e));
            c->timer.pool.push_back(e);
        }
    }
    return E2S_OK;
}

int e2s_ctx_kernel_time(e2s_ctx* c, int kernel, double* total_ms, uint64_t* launches) {
    if (!c || !total_ms || !launches || kernel < 0 || kernel >= E2S_KERNEL_COUNT) return fail(c, E2S_ERR_ARG, "bad argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    double ms = 0;
    uint64_t cnt = 0;
    std::vector<KernelTimer::Rec> keep;
    for (auto& r : c->timer.recs) {
        if (r.id != kernel) {
            keep.push_back(r);
            continue;
        }
        float t = 0;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) {
            ms += t;
            ++cnt;
        }
        c->timer.give(r.a);
        c->timer.give(r.b);
    }
    c->timer.recs.swap(keep);
    *total_ms = ms;
    *launches = cnt;
    return E2S_OK;
}

int e2s_ctx_mem_info(e2s_ctx* c, uint64_t* free_bytes, uint64_t* total_bytes) {
    if (!c) return fail(nullptr, E2S_ERR_ARG, "ctx == NULL");
    CU(c, cudaSetDevice(c->device));
    size_t f = 0, t = 0;
    CU(c, cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    return E2S_OK;
}

// ---------------------------------------------------------------------------------------------
// one process per GPU: the inter-phase exchange inside the library (NCCL on the context's stream)
// ---------------------------------------------------------------------------------------------
int e2s_comm_unique_id(uint8_t* id128) {
    if (!id128) return fail(nullptr, E2S_ERR_ARG, "e2s_comm_unique_id: NULL argument");
    NcclApi* na = nccl_api();
    if (!na) return fail(nullptr, E2S_ERR_UNSUPPORTED, "libnccl.so.2 not found");
    e2s_nccl_id id;
    const int r = na->GetUniqueId(&id);
    if (r != 0) return fail(nullptr, E2S_ERR_CUDA, std::string("ncclGetUniqueId: ") + (na->GetErrorString ? na->GetErrorString(r) : "error"));
    memcpy(id128, id.internal, 128);
    return E2S_OK;
}

int e2s_comm_create(e2s_ctx* c, const uint8_t* id128, int rank, int world, e2s_comm** out) {
    if (!c || !id128 || !out || world < 1 || rank < 0 || rank >= world) return fail(c, E2S_ERR_ARG, "e2s_comm_create: bad argument");
    *out = nullptr;
    NcclApi* na = nccl_api();
    if (!na) return fail(c, E2S_ERR_UNSUPPORTED, "libnccl.so.2 not found");
    CU(c, cudaSetDevice(c->device));
    e2s_comm* cm = new e2s_comm();
    cm->ctx = c;
    cm->rank = rank;
    cm->world = world;
    e2s_nccl_id id;
    memcpy(id.internal, id128, 128);
    const int r = na->CommInitRank(&cm->nccl, world, id, rank);
    if (r != 0) {
        delete cm;
        return fail(c, E2S_ERR_CUDA, std::string("ncclCommInitRank: ") + (na->GetErrorString ? na->GetErrorString(r) : "error"));
    }
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&cm->d_send), XR_WORDS * 8);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&cm->d_recv), size_t(world) * XR_WORDS * 8);
    if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&cm->h_recv), size_t(world) * XR_WORDS * 8, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        e2s_comm_destroy(cm);
        return fail(c, E2S_ERR_NOMEM, "e2s_comm_create: exchange buffers");
    }
    *out = cm;
    return E2S_OK;
}

void e2s_comm_destroy(e2s_comm* cm) {
    if (!cm) return;
    cudaSetDevice(cm->ctx->device);
    if (cm->nccl) {
        if (NcclApi* na = nccl_api()) na->CommDestroy(cm->nccl);
    }
    cudaFree(cm->d_send);
    cudaFree(cm->d_recv);
    cudaFreeHost(cm->h_recv);
    delete cm;
}

}  // extern "C"
