// C ABI (include/ebwt2snp_b200.h): contexts, shard residency, orchestration of the kernels,
// and the host-only integer logic (shard merge + tail/phantom rule, statistics loop, .snp text).

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <dlfcn.h>
#include <unistd.h>

#include <atomic>
#include <initializer_list>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "internal.h"
#include "merge.cuh"
#include "planes.cuh"

using namespace e2s;

struct e2s_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    std::string err;
    uint64_t launches = 0;
    // read collection
    uint8_t* d_bases = nullptr;
    uint64_t* d_off = nullptr;
    uint64_t n_reads = 0, n_bases = 0;
    uint64_t reads_cap_bases = 0, reads_cap_off = 0;
    bool reads_owned = false;
    uint32_t* d_reads_flag = nullptr;  // [0] bit 0: a staged base outside ACGTacgt, bit 1: a lower-case base; [1] != 0: reads of different lengths
    // staging: two raw-record buffers, the H2D copies run on their own stream ahead of the de-interleave kernels
    uint8_t* d_raw[2] = {nullptr, nullptr};
    size_t raw_cap = 0;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_unpacked[2] = {nullptr, nullptr}, ev_start = nullptr;
    uint8_t* d_soa_stage[2] = {nullptr, nullptr};  // e2s_pipeline_host_soa: lcp + BWT bytes of a chunk as they crossed PCIe
    size_t soa_stage_cap = 0;
    cudaEvent_t ev_soa_staged[2] = {nullptr, nullptr}, ev_soa_free[2] = {nullptr, nullptr};
    // e2s_shard_load_gesa_fd: ring of pinned pieces the reader threads fill from the file
    uint8_t* pin_ring = nullptr;
    size_t pin_piece = 0;  // bytes per slot
    cudaEvent_t ev_slot[4] = {nullptr, nullptr, nullptr, nullptr};
    // cached shard for e2s_pipeline_host
    e2s_shard* cached = nullptr;
    KernelTimer timer;
};

constexpr uint64_t GSA_TAIL = 512;  // lean SoA mode: text / suff of the last positions of the eBWT are loaded like the rest (phantom records, tail clusters)

struct e2s_shard {
    e2s_ctx* ctx = nullptr;
    uint64_t n_local = 0, global_off = 0, n_global = 0;
    uint64_t alloc_r = 0;  // elements available from local position 0
    uint32_t *lcp_a = nullptr, *text_a = nullptr, *suff_a = nullptr;
    uint8_t* bwt_a = nullptr;
    uint32_t *lcp = nullptr, *text = nullptr, *suff = nullptr;  // local position 0
    uint8_t* bwt = nullptr;
    uint8_t* lcpt = nullptr;     // bit-sliced copy of the LCP (k_derive: 64-byte groups of 7 bit planes + the plane A), 1 B/position
    bool lcpt_ok = false;        // the bit-sliced copy is there for the one-pass scan to stream (E2S_LCP_WIDE=1 switches it off)
    bool lcpt_sat = false;       // an LCP value the scan looks at is > 127 and was saturated to 127 in the copy: "lcp >= k" is
                                 // still exact for k <= 127 (the plane A is derived from the exact values), so only -k > 127 needs
                                 // the 4-byte stream then
    bool sealed = false;
    int lay_x = 4, lay_y = 4, lay_z = 4, lay_bcr = 0;  // layout of the index files (phantom record only)
    // record list
    uint64_t* d_start = nullptr;
    uint16_t* d_len = nullptr;
    uint64_t rec_cap = 0;
    uint64_t m_own = 0;     // records produced by the scan (or staged)
    uint64_t m_list = 0;    // records phase 2 analyses = own + adopted
    bool have_clusters = false, staged = false, finalized = false;
    e2s_cluster_merged merged;
    // scan scratch
    uint32_t* d_flags = nullptr;  // START words then END words
    uint64_t flag_words = 0;
    uint64_t* d_desc = nullptr;
    size_t desc_cap = 0;
    // one-pass scan (k_cluster_scan): one chunk of tiles per CTA, each with its own segment of the record arrays
    uint64_t* d_seg_start = nullptr;
    uint16_t* d_seg_len = nullptr;
    uint64_t seg_cap = 0;            // records per segment
    uint64_t seg_total = 0;          // records the segment arrays hold in all
    uint32_t n_chunks = 0, tiles_per_chunk = 0;
    ChunkRec* d_chunks = nullptr;    // SCAN_MAX_CHUNKS chunk summaries
    ChunkSeg* d_segs = nullptr;      // ... and where k_chunk_resolve put each segment in the position-ordered list
    bool contiguous = true;          // d_start / d_len hold the record list (false: it still lies in the segments)
    bool adopt_put = false;          // the records adopted from the merge have been appended to d_start / d_len
    bool pf_has_adopted = false;     // ... and the survivor list already holds them (k_merge_stats appended them)
    bool last_one_pass = false;      // what the last scan used
    uint64_t pf_want = 0;            // survivor-list capacity asked for after an overflow
    uint64_t* d_row = nullptr;       // this shard's exchange row (XR_WORDS) when there is no communicator
    MergeOut* d_mout = nullptr;      // k_merge_stats output
    MergeOut* h_mout = nullptr;      // ... its pinned host copy
    ClusterDev* d_res = nullptr;
    ClusterDev h_res;           // host copy of the last scan's accumulators (incl. length histogram)
    ClusterDev* h_pin = nullptr; // pinned staging for that copy
    bool have_scan_stats = false;
    uint8_t* d_packed = nullptr;
    uint64_t packed_cap = 0;
    unsigned long long* d_hist = nullptr;
    // fused prefilter (pipeline mode): armed by e2s_pipeline_resident with clust2snp's -m before the scan
    uint32_t pf_arm = 0;             // mcov to use in the next e2s_cluster_run, 0 = plain scan
    uint32_t pf_mcov = 0;            // what the last scan used
    SurvEntry* d_pf_list = nullptr;
    uint64_t pf_cap = 0, pf_count = 0;
    bool pf_ok = false;              // the list is complete (no overflow) and belongs to the current record list
    uint4* d_planes = nullptr;       // resident base-code bit planes of the BWT (planes.cuh), written by the loads
    uint32_t* d_seal_flag = nullptr; // != 0: an LCP value above 127 (set at seal)
    int variant = 0;
    // chunked mode (streaming): the device buffers hold one chunk [global_off, global_off + n_local) of the shard's range at a time
    bool chunked = false;
    // lean SoA mode (e2s_shard_host_gsa): text / suff stay on the host in the BCR pairSA layout; only the records of the clusters
    // that reach phase 2 are fetched from there (capture_survivors), the last GSA_TAIL positions of the eBWT excepted
    const uint8_t* host_gsa = nullptr;
    int gsa_y = 4, gsa_z = 4;
    uint64_t lean_h2d = 0, lean_d2h = 0;                    // bytes of the survivor fetches (for the callers' accounting)
    SnpDev* d_stage_dev = nullptr;                           // e2s_chunk_stage_clusters: K3a's counters
    SurvEntry* h_surv = nullptr; size_t h_surv_cap = 0;     // pinned
    uint32_t* h_gather = nullptr; size_t h_gather_cap = 0;  // pinned: text values then suff values of one capture
    uint64_t range_lo = 0, range_n = 0;   // the shard's own range of the eBWT
    uint64_t chunk_cap = 0;               // positions the buffers hold
    bool chunk_open = false;              // a chunk has been begun and not yet scanned
    bool records_flushed = false;         // e2s_chunked_finish ran: the records were handed out chunk by chunk
    ClusterDev acc;                       // the range's accumulators so far (host)
    uint64_t carry_state = 0;             // open-cluster state after the chunks so far: 0 closed, 1 unknown (an earlier shard decides), >= 2: 2 + global START
    uint32_t* p_lcp = nullptr;            // payload of the surviving clusters (see CaptureParams)
    uint32_t* p_text = nullptr;
    uint32_t* p_suff = nullptr;
    uint8_t* p_bwt = nullptr;
    uint64_t pay_cap = 0, pay_used = 0;
    SurvEntry* d_surv = nullptr;
    uint64_t surv_cap = 0, surv_count = 0;
    unsigned long long* d_cap_counters = nullptr;  // payload cursor, survivor count, error bits
    // phase 2
    SnpWork* work = nullptr;
    std::vector<e2s_event> events;
    uint64_t n_variants = 0;
    bool have_events = false, events_expanded = false;
};

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


struct e2s_comm {
    e2s_ctx* ctx = nullptr;
    void* nccl = nullptr;
    int rank = 0, world = 1;
    uint64_t* d_send = nullptr;  // XR_WORDS
    uint64_t* d_recv = nullptr;  // world * XR_WORDS
    uint64_t* h_recv = nullptr;  // pinned
};

static thread_local std::string g_err;

static int fail(e2s_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    g_err = msg;
    return code;
}
static int cuda_fail(e2s_ctx* ctx, cudaError_t e, const char* what) {
    return fail(ctx, E2S_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(ctx, x)                                      \
    do {                                                \
        cudaError_t _e = (x);                           \
        if (_e != cudaSuccess) return cuda_fail(ctx, _e, #x); \
    } while (0)

// every field of an index record is 1, 2, 4 or 8 bytes wide
static int check_field_sizes(e2s_ctx* c, std::initializer_list<int> sizes) {
    for (int v : sizes)
        if (!(v == 1 || v == 2 || v == 4 || v == 8)) return fail(c, E2S_ERR_ARG, "field byte sizes must be 1, 2, 4 or 8");
    return E2S_OK;
}

// one record of a .clusters file: 8-byte start, 2-byte length
static void put_rec10(uint8_t* o, uint64_t start, uint64_t len) {
    const uint16_t l16 = uint16_t(len);
    memcpy(o, &start, 8);
    memcpy(o + 8, &l16, 2);
}
static void get_rec10(const uint8_t* r, uint64_t* start, uint16_t* len) {
    memcpy(start, r, 8);
    memcpy(len, r + 8, 2);
}

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

// ---------------------------------------------------------------------------------------------
// shard residency
// ---------------------------------------------------------------------------------------------
static uint64_t round_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// buf = positions the device buffers hold: the whole range (resident shard) or one chunk of it (chunked shard)
static int shard_create_impl(e2s_ctx* c, uint64_t n_local, uint64_t global_off, uint64_t n_global, uint64_t buf, e2s_shard** out) {
    if (!c || !out) return fail(c, E2S_ERR_ARG, "e2s_shard_create: NULL argument");
    *out = nullptr;
    if (n_local < 2 || global_off + n_local > n_global || (global_off != 0 && global_off < 2))
        return fail(c, E2S_ERR_ARG, "e2s_shard_create: need n_local >= 2 and a range inside [0, n_global)");
    if (n_global >= (uint64_t(1) << 47)) return fail(c, E2S_ERR_UNSUPPORTED, "e2s_shard_create: n_global must be < 2^47 positions");
    CU(c, cudaSetDevice(c->device));
    e2s_shard* s = new e2s_shard();
    s->ctx = c;
    s->n_local = n_local;
    s->global_off = global_off;
    s->n_global = n_global;
    s->alloc_r = round_up(buf, 32768) + 8192;  // whole K2 tiles (32768 positions) + one K1 tile of slack
    const size_t ne = size_t(PAD_L) + s->alloc_r;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->lcp_a), ne * 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->text_a), ne * 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->suff_a), ne * 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->bwt_a), ne);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_res), sizeof(ClusterDev));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_hist), (E2S_HIST_BINS + 1) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_seal_flag), 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_planes), plane_quads(s->alloc_r) * sizeof(uint4));
    if (e != cudaSuccess) {
        e2s_shard_destroy(s);
        return fail(c, E2S_ERR_NOMEM, std::string("shard allocation: ") + cudaGetErrorString(e));
    }
    // the bit-sliced copy of the LCP the one-pass scan streams (1 B/position); without room for it the shard stays on the 4-byte stream
    if (cudaMalloc(reinterpret_cast<void**>(&s->lcpt), lcpt_bytes(s->alloc_r)) != cudaSuccess) {
        cudaGetLastError();
        s->lcpt = nullptr;
    }
    if (s->lcpt) CU(c, cudaMemsetAsync(s->lcpt, 0, lcpt_bytes(s->alloc_r), c->stream));
    CU(c, cudaMemsetAsync(s->d_planes, 0, plane_quads(s->alloc_r) * sizeof(uint4), c->stream));  // pads: code 0
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));
    s->lcp = s->lcp_a + PAD_L;
    s->text = s->text_a + PAD_L;
    s->suff = s->suff_a + PAD_L;
    s->bwt = s->bwt_a + PAD_L;
    // only the pads need defined contents (left halo of shard 0 = 0; right pad is read, never used)
    CU(c, cudaMemsetAsync(s->lcp_a, 0, PAD_L * 4, c->stream));
    CU(c, cudaMemsetAsync(s->text_a, 0, PAD_L * 4, c->stream));
    CU(c, cudaMemsetAsync(s->suff_a, 0, PAD_L * 4, c->stream));
    CU(c, cudaMemsetAsync(s->bwt_a, 0, PAD_L, c->stream));
    const size_t tail = size_t(s->alloc_r - buf);
    CU(c, cudaMemsetAsync(s->lcp + buf, 0, tail * 4, c->stream));
    CU(c, cudaMemsetAsync(s->text + buf, 0, tail * 4, c->stream));
    CU(c, cudaMemsetAsync(s->suff + buf, 0, tail * 4, c->stream));
    CU(c, cudaMemsetAsync(s->bwt + buf, 0, tail, c->stream));
    s->work = snp_work_create();
    *out = s;
    return E2S_OK;
}

int e2s_shard_create(e2s_ctx* c, uint64_t n_local, uint64_t global_off, uint64_t n_global, e2s_shard** out) {
    return shard_create_impl(c, n_local, global_off, n_global, n_local, out);
}

// ---------------------------------------------------------------------------------------------
// chunked shards (streaming): a chunk is a shard in time
// ---------------------------------------------------------------------------------------------
// positions the buffers of a chunked shard over n_local positions hold when chunk_positions are asked for
static uint64_t chunk_buffer_positions(uint64_t chunk_positions, uint64_t n_local) {
    if (chunk_positions < 16384) chunk_positions = 16384;
    chunk_positions = round_up(chunk_positions, 16384);  // chunks start at whole scan tiles
    return chunk_positions < round_up(n_local, 16384) ? chunk_positions : round_up(n_local, 16384);
}

int e2s_shard_create_chunked(e2s_ctx* c, uint64_t n_local, uint64_t global_off, uint64_t n_global, uint64_t chunk_positions,
                             e2s_shard** out) {
    const uint64_t cap = chunk_buffer_positions(chunk_positions, n_local);
    int rc = shard_create_impl(c, n_local, global_off, n_global, cap, out);
    if (rc) return rc;
    e2s_shard* s = *out;
    s->chunked = true;
    s->range_lo = global_off;
    s->range_n = n_local;
    s->chunk_cap = cap;
    memset(&s->acc, 0, sizeof s->acc);
    s->carry_state = global_off == 0 ? 0 : 1;
    if (cudaMalloc(reinterpret_cast<void**>(&s->d_cap_counters), 4 * 8) != cudaSuccess) {
        e2s_shard_destroy(s);
        *out = nullptr;
        return fail(c, E2S_ERR_NOMEM, "chunked shard counters");
    }
    CU(c, cudaMemsetAsync(s->d_cap_counters, 0, 4 * 8, c->stream));
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

uint64_t e2s_shard_chunk_positions(const e2s_shard* s) { return s && s->chunked ? s->chunk_cap : 0; }

// The next chunk [chunk_lo, chunk_lo + chunk_n) of the shard's range: chunks follow each other without gaps, every chunk but
// the last holds e2s_shard_chunk_positions() positions.  The loads that follow (e2s_shard_load_gesa / _soa / _soa_dev, global
// positions as always) should cover [chunk_lo - 176, chunk_lo + chunk_n + 1) as far as the eBWT reaches -- on the shard's last
// chunk + 151 as for every shard; what lies outside is ignored.
int e2s_chunk_begin(e2s_shard* s, uint64_t chunk_lo, uint64_t chunk_n) {
    if (!s || !s->chunked) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunk_begin: not a chunked shard");
    e2s_ctx* c = s->ctx;
    const uint64_t done = s->chunk_open || s->acc.ticket ? s->global_off + s->n_local : s->range_lo;  // (acc.ticket counts the chunks scanned)
    if (s->chunk_open) return fail(c, E2S_ERR_STATE, "e2s_chunk_begin: the previous chunk has not been scanned");
    if (chunk_lo != done || chunk_n < 1 || chunk_n > s->chunk_cap || chunk_lo + chunk_n > s->range_lo + s->range_n)
        return fail(c, E2S_ERR_ARG, "e2s_chunk_begin: chunks must follow each other and fit the buffers");
    if (chunk_lo + chunk_n < s->range_lo + s->range_n && chunk_n != s->chunk_cap)
        return fail(c, E2S_ERR_ARG, "e2s_chunk_begin: only the last chunk may be shorter than e2s_shard_chunk_positions()");
    CU(c, cudaSetDevice(c->device));
    s->global_off = chunk_lo;
    s->n_local = chunk_n;
    s->sealed = false;
    s->chunk_open = true;
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));
    if (chunk_lo < uint64_t(PAD_L)) {  // no (or a short) left context: the pad must read as zeros
        CU(c, cudaMemsetAsync(s->lcp_a, 0, PAD_L * 4, c->stream));
        CU(c, cudaMemsetAsync(s->text_a, 0, PAD_L * 4, c->stream));
        CU(c, cudaMemsetAsync(s->suff_a, 0, PAD_L * 4, c->stream));
        CU(c, cudaMemsetAsync(s->bwt_a, 0, PAD_L, c->stream));
        if (s->lcpt) CU(c, cudaMemsetAsync(s->lcpt, 0, LCPT_BLOCK, c->stream));
        CU(c, cudaMemsetAsync(s->d_planes, 0, (PL_PAD / 64) * sizeof(uint4), c->stream));
    }
    return E2S_OK;
}


void e2s_shard_destroy(e2s_shard* s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaFree(s->lcp_a);
    cudaFree(s->text_a);
    cudaFree(s->suff_a);
    cudaFree(s->bwt_a);
    cudaFree(s->lcpt);
    cudaFree(s->d_stage_dev);
    if (s->h_surv) cudaFreeHost(s->h_surv);
    if (s->h_gather) cudaFreeHost(s->h_gather);
    cudaFree(s->d_start);
    cudaFree(s->d_len);
    cudaFree(s->d_desc);
    cudaFree(s->d_row);
    cudaFree(s->d_mout);
    cudaFreeHost(s->h_mout);
    cudaFree(s->p_lcp);
    cudaFree(s->p_text);
    cudaFree(s->p_suff);
    cudaFree(s->p_bwt);
    cudaFree(s->d_surv);
    cudaFree(s->d_cap_counters);
    cudaFree(s->d_seg_start);
    cudaFree(s->d_seg_len);
    cudaFree(s->d_chunks);
    cudaFree(s->d_segs);
    cudaFree(s->d_flags);
    cudaFree(s->d_packed);
    cudaFreeHost(s->h_pin);
    cudaFree(s->d_res);
    cudaFree(s->d_hist);
    cudaFree(s->d_seal_flag);
    cudaFree(s->d_planes);
    cudaFree(s->d_pf_list);
    snp_work_destroy(s->work);
    if (s->ctx->cached == s) s->ctx->cached = nullptr;
    delete s;
}

// [first, first + count) clamped to the global range a shard keeps (2 positions of left halo, MAX_C_LEN + 1 of right halo) into
// [*a, *b); false when nothing of it is kept
static bool kept_span(const e2s_shard* s, uint64_t first, uint64_t count, uint64_t* a, uint64_t* b) {
    // (a chunk keeps PAD_L positions of left context: clusters that end in it may start up to 150 positions before it)
    const uint64_t left = s->chunked ? uint64_t(PAD_L) : 2;
    const uint64_t lo = s->global_off >= left ? s->global_off - left : 0;
    const uint64_t h = s->global_off + s->n_local + MAX_C_LEN + 1;
    const uint64_t hi = h < s->n_global ? h : s->n_global;
    *a = first > lo ? first : lo;
    *b = first + count < hi ? first + count : hi;
    return *a < *b;
}

// the two raw-record staging buffers of the loads hold at least `need` bytes each
static int ensure_raw(e2s_ctx* c, size_t need) {
    if (need <= c->raw_cap) return E2S_OK;
    CU(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 2; ++i) {
        cudaFree(c->d_raw[i]);
        c->d_raw[i] = nullptr;
    }
    c->raw_cap = 0;
    for (int i = 0; i < 2; ++i)
        if (cudaMalloc(reinterpret_cast<void**>(&c->d_raw[i]), need) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "raw staging buffer");
    c->raw_cap = need;
    return E2S_OK;
}

// the copy stream and the events every user of it shares (each is made when first missing, whichever user comes first)
static int ensure_copy_stream(e2s_ctx* c) {
    if (!c->copy_stream) CU(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        if (!c->ev_copied[i]) CU(c, cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
        if (!c->ev_unpacked[i]) CU(c, cudaEventCreateWithFlags(&c->ev_unpacked[i], cudaEventDisableTiming));
    }
    if (!c->ev_start) CU(c, cudaEventCreateWithFlags(&c->ev_start, cudaEventDisableTiming));
    return E2S_OK;
}

// the scan looks at positions [-2, n_local] (on the last shard lcp[n_local] is the phantom, which only feeds END(n-1),
// left to the host tail rule): only those decide whether the byte copy is usable
static int64_t checked_hi(const e2s_shard* s) { return int64_t(s->n_local) + (s->global_off + s->n_local == s->n_global ? 0 : 1); }

// every load also writes the narrow resident copies of what it loaded (k_derive): byte LCP + base-code bit planes
static cudaError_t derive_loaded(e2s_shard* s, int64_t l, uint64_t cnt, bool have_lcp, bool have_bwt) {
    return launch_derive(s->lcp, have_bwt ? s->bwt : nullptr, have_lcp ? s->lcpt : nullptr, s->d_planes,
                         l, l + int64_t(cnt), -2, checked_hi(s), s->d_seal_flag, s->ctx->stream, s->ctx->sm_count);
}

// Called once per LCP load with the global positions [a, b) the whole call writes, before its first piece: a load over all the
// checked positions (left of global position 0 there is only the zero pad) replaces every value the last verdict came from, so
// a reloaded shard forgets it.  A partial reload keeps it (conservative: the 4-byte stream, still exact).
static cudaError_t forget_verdict_if_covered(e2s_shard* s, uint64_t a, uint64_t b) {
    const int64_t chk_lo = s->global_off >= 2 ? -2 : -int64_t(s->global_off);
    if (int64_t(a) - int64_t(s->global_off) > chk_lo || int64_t(b) - int64_t(s->global_off) < checked_hi(s)) return cudaSuccess;
    return cudaMemsetAsync(s->d_seal_flag, 0, 4, s->ctx->stream);
}

int e2s_shard_load_gesa(e2s_shard* s, const void* records, uint64_t first, uint64_t count, int x, int y, int z) {
    if (!s || !records) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_gesa: NULL argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    CU(c, cudaSetDevice(c->device));
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = 0;
    CU(c, forget_verdict_if_covered(s, a, b));
    const int rs = x + y + z + 1;
    const uint64_t chunk = uint64_t(1) << 22;  // records per H2D chunk (multiple of 16)
    if ((rc = ensure_raw(c, size_t(chunk < (b - a) ? chunk : round_up(b - a, 16)) * rs + 64))) return rc;
    if ((rc = ensure_copy_stream(c))) return rc;
    // the copy stream starts after everything already queued on the context's stream (earlier unpack kernels read d_raw)
    CU(c, cudaEventRecord(c->ev_start, c->stream));
    CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_start, 0));
    const uint8_t* src = static_cast<const uint8_t*>(records);
    uint64_t i = 0;
    for (uint64_t p = a; p < b; p += chunk, ++i) {
        const uint64_t cnt = b - p < chunk ? b - p : chunk;
        const int buf = int(i & 1);
        if (i >= 2) CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_unpacked[buf], 0));  // the kernel that read this buffer is done
        CU(c, cudaMemcpyAsync(c->d_raw[buf], src + (p - first) * rs, size_t(cnt) * rs, cudaMemcpyHostToDevice, c->copy_stream));
        CU(c, cudaEventRecord(c->ev_copied[buf], c->copy_stream));
        CU(c, cudaStreamWaitEvent(c->stream, c->ev_copied[buf], 0));
        const int64_t l = int64_t(p) - int64_t(s->global_off);  // local index, may be -2 / -1
        CU(c, launch_unpack_gesa(c->d_raw[buf], cnt, x, y, z, s->lcp + l, s->text + l, s->suff + l, s->bwt + l, c->stream, c->sm_count));
        CU(c, cudaEventRecord(c->ev_unpacked[buf], c->stream));
        CU(c, derive_loaded(s, l, cnt, true, true));
        c->launches += 2;
    }
    s->sealed = false;
    return E2S_OK;
}

// The same straight from the file (what egsa_stream does, ref:include.hpp:42-81,120-155, instead of one istream::read per
// field): reader threads pread() pieces of the file into a ring of pinned buffers while the copy engine moves the pieces
// before them and the de-interleave kernel unpacks the ones before those.  Record i of the file = global position i.
int e2s_shard_load_gesa_fd(e2s_shard* s, int fd, uint64_t first, uint64_t count, int x, int y, int z) {
    if (!s || fd < 0) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_gesa_fd: bad argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    CU(c, cudaSetDevice(c->device));
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = 0;
    CU(c, forget_verdict_if_covered(s, a, b));
    const int rs = x + y + z + 1;
    constexpr int R = 4;                          // pinned slots
    const uint64_t piece = uint64_t(1) << 20;     // records per piece (multiple of 16)
    const size_t piece_bytes = size_t(piece) * rs + 64;
    if (c->pin_piece < piece_bytes) {
        CU(c, cudaStreamSynchronize(c->stream));
        if (c->pin_ring) cudaFreeHost(c->pin_ring);
        c->pin_ring = nullptr;
        c->pin_piece = 0;
        if (cudaHostAlloc(reinterpret_cast<void**>(&c->pin_ring), piece_bytes * R, cudaHostAllocDefault) != cudaSuccess)
            return fail(c, E2S_ERR_NOMEM, "pinned read ring");
        c->pin_piece = piece_bytes;
    }
    if ((rc = ensure_raw(c, piece_bytes))) return rc;
    if ((rc = ensure_copy_stream(c))) return rc;
    for (int i = 0; i < R; ++i)
        if (!c->ev_slot[i]) CU(c, cudaEventCreateWithFlags(&c->ev_slot[i], cudaEventDisableTiming));
    CU(c, cudaEventRecord(c->ev_start, c->stream));
    CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_start, 0));

    const uint64_t n_pieces = (b - a + piece - 1) / piece;
    std::atomic<int64_t> filled(-1), recorded(-1);  // last piece read from the file / last piece whose copy has been enqueued
    std::atomic<int> stop(0), read_err(0);
    int env_threads = 6;
    if (const char* e = getenv("E2S_READ_THREADS")) env_threads = atoi(e) > 0 ? atoi(e) : 6;
    const int T = env_threads > 16 ? 16 : env_threads;
    const int device = c->device;
    std::thread filler([&]() {
        cudaSetDevice(device);
        for (uint64_t p = 0; p < n_pieces && !stop.load(); ++p) {
            const int slot = int(p % R);
            if (p >= uint64_t(R)) {  // the copy that last read this slot must be over
                while (recorded.load(std::memory_order_acquire) < int64_t(p) - R && !stop.load()) std::this_thread::yield();
                if (stop.load()) break;
                cudaEventSynchronize(c->ev_slot[slot]);
            }
            const uint64_t p0 = a + p * piece, cnt = b - p0 < piece ? b - p0 : piece;
            uint8_t* dst = c->pin_ring + size_t(slot) * c->pin_piece;
            const size_t bytes = size_t(cnt) * rs;
            const off_t off0 = off_t(p0) * rs;
            auto part = [&](int t) {  // thread t of T: its share of the piece, 4 KB granules
                size_t lo_b = (bytes * size_t(t) / size_t(T)) & ~size_t(4095), hi_b = t + 1 == T ? bytes : (bytes * size_t(t + 1) / size_t(T)) & ~size_t(4095);
                while (lo_b < hi_b) {
                    const ssize_t got = pread(fd, dst + lo_b, hi_b - lo_b, off0 + off_t(lo_b));
                    if (got <= 0) {
                        read_err.store(1);
                        return;
                    }
                    lo_b += size_t(got);
                }
            };
            std::vector<std::thread> th;
            for (int t = 1; t < T; ++t) th.emplace_back(part, t);
            part(0);
            for (auto& w : th) w.join();
            filled.store(int64_t(p), std::memory_order_release);
            if (read_err.load()) break;
        }
    });
    rc = E2S_OK;
    cudaError_t ce = cudaSuccess;
    for (uint64_t p = 0; p < n_pieces && ce == cudaSuccess; ++p) {
        while (filled.load(std::memory_order_acquire) < int64_t(p) && !read_err.load()) std::this_thread::yield();
        if (read_err.load()) {
            rc = E2S_ERR_ARG;
            break;
        }
        const int slot = int(p % R), buf = int(p & 1);
        const uint64_t p0 = a + p * piece, cnt = b - p0 < piece ? b - p0 : piece;
        if (p >= 2) ce = cudaStreamWaitEvent(c->copy_stream, c->ev_unpacked[buf], 0);  // the kernel that read this device buffer is done
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(c->d_raw[buf], c->pin_ring + size_t(slot) * c->pin_piece, size_t(cnt) * rs, cudaMemcpyHostToDevice, c->copy_stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->ev_copied[buf], c->copy_stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->ev_slot[slot], c->copy_stream);
        recorded.store(int64_t(p), std::memory_order_release);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(c->stream, c->ev_copied[buf], 0);
        const int64_t l = int64_t(p0) - int64_t(s->global_off);  // local index, may be negative (left context)
        if (ce == cudaSuccess) ce = launch_unpack_gesa(c->d_raw[buf], cnt, x, y, z, s->lcp + l, s->text + l, s->suff + l, s->bwt + l, c->stream, c->sm_count);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->ev_unpacked[buf], c->stream);
        if (ce == cudaSuccess) ce = derive_loaded(s, l, cnt, true, true);
        c->launches += 2;
    }
    stop.store(1);
    filler.join();
    // the ring is reused by the next call: its last copies must have left it
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->copy_stream);
    s->sealed = false;
    if (ce != cudaSuccess) return cuda_fail(c, ce, "e2s_shard_load_gesa_fd");
    if (rc) return fail(c, rc, "e2s_shard_load_gesa_fd: short read from the index file");
    return E2S_OK;
}

static int load_soa(e2s_shard* s, const uint32_t* lcp, const uint32_t* text, const uint32_t* suff, const uint8_t* bwt,
                    uint64_t first, uint64_t count, cudaMemcpyKind kind) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    const int64_t l = int64_t(a) - int64_t(s->global_off);
    const uint64_t so = a - first, cnt = b - a;
    if (lcp) CU(c, forget_verdict_if_covered(s, a, b));
    if (lcp) CU(c, cudaMemcpyAsync(s->lcp + l, lcp + so, cnt * 4, kind, c->stream));
    if (text) CU(c, cudaMemcpyAsync(s->text + l, text + so, cnt * 4, kind, c->stream));
    if (suff) CU(c, cudaMemcpyAsync(s->suff + l, suff + so, cnt * 4, kind, c->stream));
    if (bwt) CU(c, cudaMemcpyAsync(s->bwt + l, bwt + so, cnt, kind, c->stream));
    if (lcp || bwt) {
        CU(c, derive_loaded(s, l, cnt, lcp != nullptr, bwt != nullptr));
        ++c->launches;
    }
    s->sealed = false;
    return E2S_OK;
}

int e2s_shard_load_soa(e2s_shard* s, const uint32_t* lcp, const uint32_t* text, const uint32_t* suff, const uint8_t* bwt,
                       uint64_t first, uint64_t count) {
    return load_soa(s, lcp, text, suff, bwt, first, count, cudaMemcpyHostToDevice);
}
int e2s_shard_load_soa_dev(e2s_shard* s, const uint32_t* lcp, const uint32_t* text, const uint32_t* suff,
                           const uint8_t* bwt, uint64_t first, uint64_t count) {
    return load_soa(s, lcp, text, suff, bwt, first, count, cudaMemcpyDeviceToDevice);
}

// ---- lean SoA inputs (the BCR triple: X.out.lcp, X.out, X.out.pairSA; ref:include.hpp:157-188) -----------------------------
// Phase 1 and the prefilter need the LCP and the BWT only: 1 + x bytes per position cross PCIe instead of the 13 of an EGSA
// record.  text / suff (the pairSA file) stay on the host; the records of the ~0.1 % of the clusters that reach phase 2 are
// fetched from there when a chunk's survivors are captured.
int e2s_shard_host_gsa(e2s_shard* s, const void* pair_sa, int y, int z) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (!s->chunked) return fail(s->ctx, E2S_ERR_STATE, "e2s_shard_host_gsa: chunked shards only (the survivors' records are captured per chunk)");
    if (pair_sa)
        if (int rc = check_field_sizes(s->ctx, {y, z})) return rc;
    s->host_gsa = static_cast<const uint8_t*>(pair_sa);
    s->gsa_y = y;
    s->gsa_z = z;
    return E2S_OK;
}

// the text / suff of the last GSA_TAIL positions of the eBWT, as far as [a, b) holds them: the phantom records past EOF are made
// of them, and clusters that start there are captured from the device
static int lean_load_tail(e2s_shard* s, uint64_t a, uint64_t b) {
    e2s_ctx* c = s->ctx;
    if (!s->host_gsa) return E2S_OK;
    const uint64_t tail_lo = s->n_global > GSA_TAIL ? s->n_global - GSA_TAIL : 0;
    const uint64_t ta = a > tail_lo ? a : tail_lo;
    if (ta >= b) return E2S_OK;
    std::vector<uint32_t> t(size_t(b - ta)), sf(size_t(b - ta));
    const int rs = s->gsa_y + s->gsa_z;
    for (uint64_t p = ta; p < b; ++p) {
        const uint8_t* g = s->host_gsa + p * uint64_t(rs);
        uint32_t vs = 0, vt = 0;
        for (int q = 0; q < (s->gsa_z < 4 ? s->gsa_z : 4); ++q) vs |= uint32_t(g[q]) << (8 * q);
        for (int q = 0; q < (s->gsa_y < 4 ? s->gsa_y : 4); ++q) vt |= uint32_t(g[s->gsa_z + q]) << (8 * q);
        sf[size_t(p - ta)] = vs;
        t[size_t(p - ta)] = vt;
    }
    const int64_t lt = int64_t(ta) - int64_t(s->global_off);
    CU(c, cudaMemcpyAsync(s->text + lt, t.data(), (b - ta) * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(s->suff + lt, sf.data(), (b - ta) * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));  // (the vectors go out of scope)
    return E2S_OK;
}

// lcp (x bytes per position) + BWT bytes of the global positions [first, first + count) -> the shard's resident arrays and their
// narrow copies.  dev: the sources are device memory (a staging buffer the caller filled), else host memory.
static int load_lcp_bwt(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, uint64_t first, uint64_t count, bool dev) {
    e2s_ctx* c = s->ctx;
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_x = x;
    CU(c, forget_verdict_if_covered(s, a, b));
    const uint8_t* src = static_cast<const uint8_t*>(lcp);
    const int64_t l0 = int64_t(a) - int64_t(s->global_off);
    const cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (x == 4) {  // already at the resident width
        CU(c, cudaMemcpyAsync(s->lcp + l0, src + (a - first) * 4, (b - a) * 4, kind, c->stream));
    } else if (dev) {
        CU(c, launch_widen(src + (a - first) * uint64_t(x), x, s->lcp + l0, b - a, c->stream, c->sm_count));
        ++c->launches;
    } else {
        const uint64_t piece = uint64_t(1) << 24;
        if (int rc = ensure_raw(c, size_t(piece) * x + 64)) return rc;
        for (uint64_t p = a; p < b; p += piece) {  // (one stream: the staging buffer is free again when the widening kernel has run)
            const uint64_t cnt = b - p < piece ? b - p : piece;
            CU(c, cudaMemcpyAsync(c->d_raw[0], src + (p - first) * uint64_t(x), cnt * uint64_t(x), cudaMemcpyHostToDevice, c->stream));
            CU(c, launch_widen(c->d_raw[0], x, s->lcp + (int64_t(p) - int64_t(s->global_off)), cnt, c->stream, c->sm_count));
            ++c->launches;
        }
    }
    CU(c, cudaMemcpyAsync(s->bwt + l0, bwt + (a - first), b - a, kind, c->stream));
    CU(c, derive_loaded(s, l0, b - a, true, true));
    ++c->launches;
    s->sealed = false;
    return lean_load_tail(s, a, b);
}

// The whole BCR triple of [first, first + count): lcp + BWT as above, and X.out.pairSA (suff(z) then text(y) per position,
// ref:include.hpp:157-188) copied as it is in the file and split / widened on the device.
int e2s_shard_load_bcr(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, const void* pair_sa, int y, int z, uint64_t first,
                       uint64_t count) {
    if (!s || !lcp || !bwt || !pair_sa) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_bcr: NULL argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    CU(c, cudaSetDevice(c->device));
    if ((rc = load_lcp_bwt(s, lcp, x, bwt, first, count, false))) return rc;
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_y = y; s->lay_z = z; s->lay_bcr = 1;
    const int rs = y + z;
    const uint64_t piece = uint64_t(1) << 22;
    if ((rc = ensure_raw(c, size_t(piece) * size_t(rs) + 64))) return rc;
    const uint8_t* src = static_cast<const uint8_t*>(pair_sa);
    uint64_t i = 0;
    for (uint64_t p = a; p < b; p += piece, ++i) {  // (one stream: a staging buffer is free again when the kernel that read it has run)
        const uint64_t cnt = b - p < piece ? b - p : piece;
        const int64_t l = int64_t(p) - int64_t(s->global_off);
        CU(c, cudaMemcpyAsync(c->d_raw[i & 1], src + (p - first) * uint64_t(rs), cnt * uint64_t(rs), cudaMemcpyHostToDevice, c->stream));
        CU(c, launch_widen_pairs(c->d_raw[i & 1], z, y, s->suff + l, s->text + l, cnt, c->stream, c->sm_count));
        ++c->launches;
    }
    return E2S_OK;
}

int e2s_shard_load_lcp_bwt(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, uint64_t first, uint64_t count) {
    if (!s || !lcp || !bwt) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_lcp_bwt: NULL argument");
    e2s_ctx* c = s->ctx;
    if (int rc = check_field_sizes(c, {x})) return rc;
    CU(c, cudaSetDevice(c->device));
    return load_lcp_bwt(s, lcp, x, bwt, first, count, false);
}

// R + 1 HOST offsets of a ragged collection, checked as every ragged builder entry point takes them; *longest = the longest read
static int check_offsets(e2s_ctx* c, const char* who, const uint64_t* off, uint64_t n_reads, uint32_t* longest) {
    if (off[0] != 0) return fail(c, E2S_ERR_ARG, std::string(who) + ": off[0] must be 0");
    uint32_t m = 0;
    for (uint64_t r = 0; r < n_reads; ++r) {
        if (off[r + 1] < off[r]) return fail(c, E2S_ERR_ARG, std::string(who) + ": read offsets must not decrease");
        const uint64_t l = off[r + 1] - off[r];
        if (l >= 65536) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": a read of 65536 bases or more (the keys are fixed-width: short reads only)");
        m = l > m ? uint32_t(l) : m;
    }
    if (m == 0) return fail(c, E2S_ERR_ARG, std::string(who) + ": every read is empty");
    *longest = m;
    return E2S_OK;
}

// the offsets in device memory (the caller frees *d_off after synchronising the stream)
static int upload_offsets(e2s_ctx* c, const char* who, const uint64_t* off, uint64_t n_reads, uint64_t** d_off) {
    if (cudaMalloc(reinterpret_cast<void**>(d_off), (n_reads + 1) * 8) != cudaSuccess) {
        cudaGetLastError();
        *d_off = nullptr;
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": read offsets on the device");
    }
    const cudaError_t eo = cudaMemcpyAsync(*d_off, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, c->stream);
    if (eo != cudaSuccess) {
        cudaFree(*d_off);
        *d_off = nullptr;
        return cuda_fail(c, eo, "H2D read offsets");
    }
    return E2S_OK;
}

// shared by the four whole-index builder entry points.  off = nullptr: n_reads reads of read_len bases; else n_reads + 1 HOST offsets.
static int build_egsa_common(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* off, uint64_t n_reads, uint32_t read_len,
                             uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt) {
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
    uint64_t total = n_reads * uint64_t(read_len);
    uint32_t longest = read_len;
    uint64_t* d_off = nullptr;
    if (off) {
        int rc = check_offsets(c, who, off, n_reads, &longest);
        if (rc == E2S_OK) rc = upload_offsets(c, who, off, n_reads, &d_off);
        if (rc != E2S_OK) return rc;
        total = off[n_reads];
    }
    cudaError_t e = build_egsa(d_reads, d_off, off, n_reads, longest, total, d_lcp, d_text, d_suff, d_bwt, c->stream, &c->launches);
    if (d_off) {
        cudaStreamSynchronize(c->stream);
        cudaFree(d_off);
    }
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": scratch buffers (24.5 bytes per suffix with 32-bit suffix ids, 32.5 with 64-bit ids)");
    }
    if (e == cudaErrorInvalidValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED,
                    std::string(who) + ": a read holds a base outside ACGT/acgt (N has no 2-bit code; the reference itself is "
                    "non-deterministic on N, ref:include.hpp:273) -- filter such reads first");
    }
    if (e == cudaErrorInvalidConfiguration) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": the collection is outside what one call sorts (read length < 65536, < 2^43 suffixes)");
    }
    if (e != cudaSuccess) return cuda_fail(c, e, "build_egsa");
    return E2S_OK;
}

int e2s_build_egsa_dev(e2s_ctx* c, const uint8_t* d_reads, uint64_t n_reads, uint32_t read_len, uint32_t* d_lcp, uint32_t* d_text,
                       uint32_t* d_suff, uint8_t* d_bwt) {
    if (!c || !d_reads || !d_lcp || !d_text || !d_suff || !d_bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_dev: NULL argument");
    if (n_reads == 0 || read_len == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_dev: empty read collection");
    CU(c, cudaSetDevice(c->device));
    return build_egsa_common(c, "e2s_build_egsa_dev", d_reads, nullptr, n_reads, read_len, d_lcp, d_text, d_suff, d_bwt);
}

int e2s_build_egsa_ragged_dev(e2s_ctx* c, const uint8_t* d_bases, const uint64_t* off, uint64_t n_reads, uint32_t* d_lcp, uint32_t* d_text,
                              uint32_t* d_suff, uint8_t* d_bwt) {
    if (!c || !d_bases || !off || !d_lcp || !d_text || !d_suff || !d_bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged_dev: NULL argument");
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged_dev: empty read collection");
    CU(c, cudaSetDevice(c->device));
    return build_egsa_common(c, "e2s_build_egsa_ragged_dev", d_bases, off, n_reads, 0, d_lcp, d_text, d_suff, d_bwt);
}

// one key range, both read shapes (arguments checked by the caller).  d_off == nullptr: n_reads reads of read_len bases; else n_reads + 1
// DEVICE offsets, read_len = the longest read, total = off[n_reads].
static int build_range_common(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, uint64_t n_reads, uint32_t read_len,
                              uint64_t total, uint64_t key_lo, uint64_t key_hi, uint32_t before_text, uint32_t before_suff, uint64_t capacity,
                              uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position) {
    const uint64_t before = before_text == 0xffffffffu ? ~uint64_t(0) : (uint64_t(before_text) << 32) | before_suff;
    *n_records = 0;
    *first_position = 0;
    cudaError_t e = build_egsa_range(d_reads, d_off, n_reads, read_len, total, key_lo, key_hi, before, capacity, d_lcp, d_text, d_suff, d_bwt,
                                     n_records, first_position, c->stream, &c->launches);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": scratch buffers (24.5 / 32.5 bytes per suffix of the range)");
    }
    if (e == cudaErrorInvalidPitchValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_ARG, std::string(who) + ": the key range holds more records than `capacity` (*n_records says how many)");
    }
    if (e == cudaErrorInvalidValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": a read holds a base outside ACGT/acgt");
    }
    if (e == cudaErrorInvalidConfiguration) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": the collection is outside what one call sorts");
    }
    if (e != cudaSuccess) return cuda_fail(c, e, "build_egsa_range");
    return E2S_OK;
}

int e2s_build_egsa_range_dev(e2s_ctx* c, const uint8_t* d_reads, uint64_t n_reads, uint32_t read_len, uint64_t key_lo, uint64_t key_hi,
                             uint32_t before_text, uint32_t before_suff, uint64_t capacity, uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff,
                             uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position) {
    if (!c || !d_reads || !d_lcp || !d_text || !d_suff || !d_bwt || !n_records || !first_position)
        return fail(c, E2S_ERR_ARG, "e2s_build_egsa_range_dev: NULL argument");
    if (n_reads == 0 || read_len == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_range_dev: empty read collection");
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, "e2s_build_egsa_range_dev: more than 2^32 - 1 reads (text is a 32-bit field)");
    if (key_hi != 0 && key_hi <= key_lo) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_range_dev: empty key range");
    CU(c, cudaSetDevice(c->device));
    return build_range_common(c, "e2s_build_egsa_range_dev", d_reads, nullptr, n_reads, read_len, n_reads * uint64_t(read_len), key_lo, key_hi,
                              before_text, before_suff, capacity, d_lcp, d_text, d_suff, d_bwt, n_records, first_position);
}

int e2s_build_egsa_ragged_range_dev(e2s_ctx* c, const uint8_t* d_bases, const uint64_t* off, uint64_t n_reads, uint64_t key_lo, uint64_t key_hi,
                                    uint32_t before_text, uint32_t before_suff, uint64_t capacity, uint32_t* d_lcp, uint32_t* d_text,
                                    uint32_t* d_suff, uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position) {
    const char* who = "e2s_build_egsa_ragged_range_dev";
    if (!c || !d_bases || !off || !d_lcp || !d_text || !d_suff || !d_bwt || !n_records || !first_position)
        return fail(c, E2S_ERR_ARG, std::string(who) + ": NULL argument");
    *n_records = 0;
    *first_position = 0;
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, std::string(who) + ": empty read collection");
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
    if (key_hi != 0 && key_hi <= key_lo) return fail(c, E2S_ERR_ARG, std::string(who) + ": empty key range");
    CU(c, cudaSetDevice(c->device));
    uint32_t longest = 0;
    uint64_t* d_off = nullptr;
    int rc = check_offsets(c, who, off, n_reads, &longest);
    if (rc == E2S_OK) rc = upload_offsets(c, who, off, n_reads, &d_off);
    if (rc != E2S_OK) return rc;
    rc = build_range_common(c, who, d_bases, d_off, n_reads, longest, off[n_reads], key_lo, key_hi, before_text, before_suff, capacity, d_lcp, d_text,
                            d_suff, d_bwt, n_records, first_position);
    cudaStreamSynchronize(c->stream);
    cudaFree(d_off);
    return rc;
}

// the four index arrays of the host builder entry points on the device
struct IndexArraysDev {
    uint8_t* bwt = nullptr;
    uint32_t *lcp = nullptr, *text = nullptr, *suff = nullptr;
    // room for m positions: all four arrays or none
    cudaError_t alloc(uint64_t m) {
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&bwt), m);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&lcp), m * 4);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&text), m * 4);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&suff), m * 4);
        if (e != cudaSuccess) {
            release();
            cudaGetLastError();
        }
        return e;
    }
    void release() {
        cudaFree(bwt); cudaFree(lcp); cudaFree(text); cudaFree(suff);
        bwt = nullptr;
        lcp = text = suff = nullptr;
    }
    // the first m positions to the host arrays, then a synchronisation
    cudaError_t to_host(uint32_t* h_lcp, uint32_t* h_text, uint32_t* h_suff, uint8_t* h_bwt, uint64_t m, cudaStream_t stream) const {
        cudaError_t e = cudaMemcpyAsync(h_lcp, lcp, m * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_text, text, m * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_suff, suff, m * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_bwt, bwt, m, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        return e;
    }
};

// An index that does not fit one call's device memory (outputs 13 B + scratch 24.5 / 32.5 B per suffix): the index key range by key
// range (build_range_common), every range's records copied to their place in the host arrays.  d_off == nullptr: n_reads reads of
// read_len bases; else DEVICE offsets (uploaded once for all ranges), read_len = the longest read.  A range that turns out to hold more
// than `cap` records is cut in two.  E2S_BUILD_RANGE_RECORDS=<cap> forces this path (tests).
static int build_egsa_host_ranges(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, uint64_t n_reads, uint32_t read_len,
                                  uint64_t total, uint64_t cap, uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt) {
    const char* range_who = d_off ? "e2s_build_egsa_ragged_range_dev" : "e2s_build_egsa_range_dev";
    const uint64_t n = total + n_reads;
    IndexArraysDev d;
    if (d.alloc(cap) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, std::string(who) + ": device buffers of one key range");
    // ranges as (lo, hi) with hi = 0 for "to the end of the key space", processed in key order from a stack
    uint64_t parts = (n + cap - 1) / cap;
    parts += parts / 4 + 1;
    std::vector<std::pair<uint64_t, uint64_t>> todo;
    for (uint64_t i = parts; i-- > 0;) {
        const uint64_t lo = uint64_t((static_cast<unsigned __int128>(i) << 64) / parts);
        const uint64_t hi = i + 1 == parts ? 0 : uint64_t((static_cast<unsigned __int128>(i + 1) << 64) / parts);
        if (hi == 0 || hi > lo) todo.emplace_back(lo, hi);
    }
    uint64_t at = 0;
    uint32_t before_text = 0xffffffffu, before_suff = 0;
    int rc = E2S_OK;
    while (!todo.empty() && rc == E2S_OK) {
        const auto [lo, hi] = todo.back();
        todo.pop_back();
        uint64_t m = 0, first = 0;
        rc = build_range_common(c, range_who, d_reads, d_off, n_reads, read_len, total, lo, hi, before_text, before_suff, cap, d.lcp, d.text, d.suff,
                                d.bwt, &m, &first);
        if (rc == E2S_ERR_ARG && m > cap) {  // too many records for the buffers: two halves (a single key value cannot be cut)
            const uint64_t width = hi - lo;  // (mod 2^64: right for hi = 0 as long as lo > 0 or the range is not the whole space)
            if (width == 1 || (lo == 0 && hi == 0)) {
                rc = fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": one 32-symbol prefix is shared by more suffixes than fit the device");
                break;
            }
            const uint64_t mid = lo + (width >> 1);
            todo.emplace_back(mid, hi);
            todo.emplace_back(lo, mid);
            rc = E2S_OK;
            continue;
        }
        if (rc != E2S_OK) break;
        if (first != at || at + m > n) {
            rc = fail(c, E2S_ERR_STATE, std::string(who) + ": key ranges do not tile the index");
            break;
        }
        if (m) {
            const cudaError_t e = d.to_host(lcp + at, text + at, suff + at, bwt + at, m, c->stream);
            if (e != cudaSuccess) {
                rc = cuda_fail(c, e, "D2H index arrays of a key range");
                break;
            }
            at += m;
            before_text = text[at - 1];
            before_suff = suff[at - 1];
        }
    }
    if (rc == E2S_OK && at != n) rc = fail(c, E2S_ERR_STATE, std::string(who) + ": key ranges do not cover the index");
    d.release();
    return rc;
}

// host buffers in and out: device buffers allocated and released here
static int build_egsa_host(e2s_ctx* c, const char* who, const uint8_t* reads, const uint64_t* off, uint64_t n_reads, uint32_t read_len,
                           uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt) {
    CU(c, cudaSetDevice(c->device));
    const uint64_t total = off ? off[n_reads] : n_reads * uint64_t(read_len);
    const uint64_t n = total + n_reads;
    // suffix ids are 64-bit beyond 2^32 (equal lengths: n; ragged: R << shift, shift = the bits of the longest read's length + 1)
    bool ids64 = n > 0xffffffffull;
    uint32_t longest = read_len;
    if (off) {
        if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
        const int rc = check_offsets(c, who, off, n_reads, &longest);
        if (rc != E2S_OK) return rc;
        uint32_t bits = 1;
        while ((longest >> bits) != 0) ++bits;
        ids64 = n_reads > (uint64_t(1) << (32 - bits));
    }
    if (getenv("E2S_BUILD_IDS64")) ids64 = true;
    uint8_t* d_reads = nullptr;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d_reads), total ? total : 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": the reads on the device");
    }
    {   // does the whole index fit one call?  13 B of outputs + up to 32.5 B of scratch per suffix, packed reads and slack (half a byte
        // per base), and for ragged reads the 2 extra packed words and the device offset of every read; the reads are already resident
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const uint64_t per_suffix = 13 + (ids64 ? 33 : 25);
        const double fixed = double(total) / 2 + (off ? 24.0 * double(n_reads) : 0.0);
        uint64_t cap = 0;
        if (const char* f = getenv("E2S_BUILD_RANGE_RECORDS")) cap = strtoull(f, nullptr, 10);
        else if (double(n) * double(per_suffix) + fixed > 0.92 * double(free_b)) {
            const double room = 0.92 * double(free_b) - fixed - double(n) / 512;
            cap = room > 0 ? uint64_t(room / double(per_suffix)) : 0;
            if (cap < 4096) {
                cudaFree(d_reads);
                return fail(c, E2S_ERR_NOMEM, std::string(who) + ": not even one key range of the index fits the device");
            }
        }
        if (cap) {
            uint64_t* d_off = nullptr;
            int rc = E2S_OK;
            if (off) rc = upload_offsets(c, who, off, n_reads, &d_off);
            if (rc == E2S_OK) {
                e = cudaMemcpyAsync(d_reads, reads, total, cudaMemcpyHostToDevice, c->stream);
                rc = e == cudaSuccess ? build_egsa_host_ranges(c, who, d_reads, d_off, n_reads, longest, total, cap, lcp, text, suff, bwt)
                                      : cuda_fail(c, e, "H2D reads");
            }
            cudaStreamSynchronize(c->stream);
            cudaFree(d_off);
            cudaFree(d_reads);
            return rc;
        }
    }
    IndexArraysDev d;
    if (d.alloc(n) != cudaSuccess) {
        cudaFree(d_reads);
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": device buffers");
    }
    e = cudaMemcpyAsync(d_reads, reads, total, cudaMemcpyHostToDevice, c->stream);
    int rc = e == cudaSuccess ? build_egsa_common(c, who, d_reads, off, n_reads, read_len, d.lcp, d.text, d.suff, d.bwt) : cuda_fail(c, e, "H2D reads");
    if (rc == E2S_OK && (e = d.to_host(lcp, text, suff, bwt, n, c->stream)) != cudaSuccess) rc = cuda_fail(c, e, "D2H index arrays");
    cudaFree(d_reads);
    d.release();
    return rc;
}

int e2s_build_egsa(e2s_ctx* c, const uint8_t* reads, uint64_t n_reads, uint32_t read_len, uint32_t* lcp, uint32_t* text, uint32_t* suff,
                   uint8_t* bwt) {
    if (!c || !reads || !lcp || !text || !suff || !bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa: NULL argument");
    if (n_reads == 0 || read_len == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa: empty read collection");
    return build_egsa_host(c, "e2s_build_egsa", reads, nullptr, n_reads, read_len, lcp, text, suff, bwt);
}

int e2s_build_egsa_ragged(e2s_ctx* c, const uint8_t* bases, const uint64_t* off, uint64_t n_reads, uint32_t* lcp, uint32_t* text,
                          uint32_t* suff, uint8_t* bwt) {
    if (!c || !bases || !off || !lcp || !text || !suff || !bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged: NULL argument");
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged: empty read collection");
    return build_egsa_host(c, "e2s_build_egsa_ragged", bases, off, n_reads, 0, lcp, text, suff, bwt);
}

int e2s_shard_set_layout(e2s_shard* s, int x, int y, int z, int bcr) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (int rc = check_field_sizes(s->ctx, {x, y, z})) return rc;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = bcr ? 1 : 0;
    s->sealed = false;
    return E2S_OK;
}

int e2s_shard_seal(e2s_shard* s) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    if (s->global_off + s->n_local == s->n_global) {  // the records past EOF (a 1-block kernel) and their narrow copies
        CU(c, launch_fill_phantom(s->lcp, s->text, s->suff, s->bwt, s->n_local, HALO_R, s->lay_x, s->lay_y, s->lay_z,
                                  s->lay_bcr, c->stream));
        CU(c, derive_loaded(s, int64_t(s->n_local), HALO_R, true, true));
        c->launches += 2;
    }
    // The byte LCP and the bit planes were written by the loads themselves: sealing costs no pass over the data, only
    // the verdict whether every LCP value the scan looks at fits the byte copy (E2S_LCP_WIDE=1 keeps the 4-byte stream,
    // for A/B measurements and the tests)
    s->lcpt_ok = s->lcpt_sat = false;
    const char* wide = getenv("E2S_LCP_WIDE");
    if (s->lcpt && !(wide && atoi(wide) != 0)) {
        uint32_t h_flag = 1;
        CU(c, cudaMemcpyAsync(&h_flag, s->d_seal_flag, 4, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        s->lcpt_ok = true;
        s->lcpt_sat = h_flag != 0;
    }
    s->sealed = true;
    return E2S_OK;
}

int e2s_shard_lcp_bytes_resident(const e2s_shard* s) { return s ? (s->sealed && s->lcpt_ok ? 1 : 4) : 0; }

// may k_cluster_scan run on this shard with these options?  (min_len <= 33: the bit-parallel length test; the saturated
// bit-sliced LCP compares exactly against k <= 127 whatever the values, against any k when nothing was saturated)
static bool one_pass_ok(const e2s_shard* s, uint32_t k, int32_t min_len) {
    return s->sealed && s->lcpt_ok && (!s->lcpt_sat || k <= 127u) && min_len <= 33;
}

// one pass over the staged reads: does any byte fall outside ACGTacgt?  (K4's consensus then needs base_to_int's general rule)
static int reads_check(e2s_ctx* c) {
    if (!c->d_reads_flag && cudaMalloc(reinterpret_cast<void**>(&c->d_reads_flag), 8) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "reads flag");
    CU(c, cudaMemsetAsync(c->d_reads_flag, 0, 8, c->stream));
    CU(c, launch_reads_check(c->d_bases, c->n_bases, c->d_off, c->n_reads, c->d_reads_flag, c->stream, c->sm_count));
    c->launches += 2;
    return E2S_OK;
}

int e2s_reads_stage(e2s_ctx* c, const uint8_t* bases, const uint64_t* off, uint64_t n_reads) {
    if (!c || !bases || !off) return fail(c, E2S_ERR_ARG, "e2s_reads_stage: NULL argument");
    CU(c, cudaSetDevice(c->device));
    const uint64_t nb = off[n_reads];
    if (!c->reads_owned || nb + 16 > c->reads_cap_bases || (n_reads + 1) > c->reads_cap_off) {  // reuse the buffers when they fit
        if (c->reads_owned) {
            cudaFree(c->d_bases);
            cudaFree(c->d_off);
        }
        c->d_bases = nullptr;
        c->d_off = nullptr;
        c->reads_owned = true;
        c->reads_cap_bases = c->reads_cap_off = 0;
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&c->d_bases), nb + 16);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->d_off), (n_reads + 1) * 8);
        if (e != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "reads allocation");
        c->reads_cap_bases = nb + 16;
        c->reads_cap_off = n_reads + 1;
    }
    CU(c, cudaMemcpyAsync(c->d_bases, bases, nb, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(c->d_off, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    c->n_reads = n_reads;
    c->n_bases = nb;
    return reads_check(c);
}

int e2s_reads_stage_dev(e2s_ctx* c, const uint8_t* d_bases, const uint64_t* d_off, uint64_t n_reads, uint64_t n_bases) {
    if (!c || !d_bases || !d_off) return fail(c, E2S_ERR_ARG, "e2s_reads_stage_dev: NULL argument");
    if (c->reads_owned) {
        cudaFree(c->d_bases);
        cudaFree(c->d_off);
    }
    c->reads_owned = false;
    c->reads_cap_bases = c->reads_cap_off = 0;
    c->d_bases = const_cast<uint8_t*>(d_bases);
    c->d_off = const_cast<uint64_t*>(d_off);
    c->n_reads = n_reads;
    c->n_bases = n_bases;
    return reads_check(c);
}

// ---------------------------------------------------------------------------------------------
// phase 1
// ---------------------------------------------------------------------------------------------
static int ensure_records(e2s_shard* s, uint64_t cap) {
    if (cap <= s->rec_cap && s->d_start) return E2S_OK;
    cudaFree(s->d_start);
    cudaFree(s->d_len);
    s->d_start = nullptr;
    s->d_len = nullptr;
    s->rec_cap = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&s->d_start), cap * 8);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_len), cap * 2 + 16);
    if (e != cudaSuccess) return fail(s->ctx, E2S_ERR_NOMEM, "cluster record buffers");
    s->rec_cap = cap;
    return E2S_OK;
}

static int ensure_segments(e2s_shard* s, uint64_t seg_cap) {
    if (seg_cap <= s->seg_cap && s->d_seg_start && seg_cap * s->n_chunks <= s->seg_total) return E2S_OK;
    cudaFree(s->d_seg_start);
    cudaFree(s->d_seg_len);
    s->d_seg_start = nullptr;
    s->d_seg_len = nullptr;
    s->seg_cap = 0;
    const size_t total = size_t(seg_cap) * s->n_chunks;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&s->d_seg_start), total * 8);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_seg_len), total * 2 + 16);
    if (e != cudaSuccess) return fail(s->ctx, E2S_ERR_NOMEM, "cluster record segments");
    s->seg_cap = seg_cap;
    s->seg_total = total;
    return E2S_OK;
}

// the position-ordered record list in d_start / d_len (the one-pass scan leaves it in per-chunk segments: exported on demand)
static int ensure_contiguous(e2s_shard* s) {
    if (s->contiguous) return E2S_OK;
    e2s_ctx* c = s->ctx;
    int rc = ensure_records(s, s->m_own + 8);
    if (rc) return rc;
    CU(c, launch_export_records(s->d_segs, s->n_chunks, s->seg_cap, s->d_seg_start, s->d_seg_len, s->d_start, s->d_len, nullptr, c->stream));
    ++c->launches;
    s->contiguous = true;
    return E2S_OK;
}

int e2s_cluster_prefilter(e2s_shard* s, int mcov_out) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (mcov_out < 0 || 2 * mcov_out > E2S_MAX_C_LEN) return fail(s->ctx, E2S_ERR_ARG, "e2s_cluster_prefilter: need 0 <= 2 * mcov_out <= 150");
    s->pf_arm = uint32_t(mcov_out);
    return E2S_OK;
}

// the summary of a shard's range [global_off, global_off + n_local) from its scan accumulators
static void make_summary(const ClusterDev& h, uint64_t n_local, uint64_t global_off, uint64_t n_global, uint32_t k, int32_t min_len,
                         uint64_t lcp_bytes, e2s_cluster_summary* sum) {
    memset(sum, 0, sizeof *sum);
    sum->n_local = n_local;
    sum->global_off = global_off;
    sum->n_global = n_global;
    sum->n_end = h.n_end;
    sum->n_written = h.n_written;
    sum->head_end = h.head_end;
    sum->any_event = h.any_event;
    sum->open_start = h.any_event ? h.open_start : 0;
    sum->end_nm2_start = h.end_nm2_start;
    sum->k = k;
    sum->min_len = uint64_t(int64_t(min_len));
    sum->lcp_bytes = lcp_bytes;
    sum->tail_lcp_nm2 = h.tail_lcp_nm2;
    sum->tail_lcp_nm1 = h.tail_lcp_nm1;
    sum->tail_bwt_nm1 = h.tail_bwt_nm1;
}

// a record segment of the one-pass scan overflowed: grow the segments to the fullest one (the chunks keep counting past their
// capacity)
static int grow_segments(e2s_shard* s) {
    std::vector<ChunkRec> hc(s->n_chunks);
    CU(s->ctx, cudaMemcpy(hc.data(), s->d_chunks, hc.size() * sizeof(ChunkRec), cudaMemcpyDeviceToHost));
    uint64_t mx = 0;
    for (const ChunkRec& r : hc) mx = r.own_count > mx ? r.own_count : mx;
    return ensure_segments(s, mx + 64);
}

// phase 2's view of the shard's resident arrays (no record list yet)
static SnpArrays shard_arrays(const e2s_shard* s) {
    SnpArrays a;
    a.lcp = s->lcp;
    a.text = s->text;
    a.suff = s->suff;
    a.bwt = s->bwt;
    a.planes = s->d_planes;
    a.n_local = s->n_local;
    a.global_off = s->global_off;
    a.cl_start = nullptr;
    a.cl_len = nullptr;
    a.m = 0;
    a.reads_flag = s->ctx->d_reads_flag;
    return a;
}

// K3a's count of length-passing clusters (2 mcov_out <= length <= max_clust_length) when the fused prefilter replaced it: from
// the scan's own length histogram and the records the shard adopted from the merge
static uint64_t analysed_count(const ClusterDev& h, const e2s_cluster_merged& mg, int mcov_out, int max_clust_length) {
    uint64_t na = 0;
    for (int l = 2 * mcov_out; l <= max_clust_length; ++l) na += h.hist[l];
    for (uint32_t i = 0; i < mg.n_adopt; ++i)
        na += int64_t(mg.adopt_len[i]) >= 2 * mcov_out && int64_t(mg.adopt_len[i]) <= max_clust_length;
    return na;
}

// every rank's exchange row (cm->d_send) into cm->d_recv, on the context's stream
static int all_gather_rows(e2s_ctx* c, e2s_comm* cm) {
    NcclApi* na = nccl_api();
    const int nr = na->AllGather(cm->d_send, cm->d_recv, XR_WORDS, NCCL_UINT64, cm->nccl, c->stream);
    if (nr != 0) return fail(c, E2S_ERR_CUDA, std::string("ncclAllGather: ") + (na->GetErrorString ? na->GetErrorString(nr) : "error"));
    return E2S_OK;
}

// K1 + K2.  cm == NULL: this shard's accumulators come back with one device-to-host copy.  cm != NULL (one process per
// GPU): the rows of ALL shards come back instead -- packed on the device, all-gathered by NCCL on the same stream, one
// copy, one synchronisation -- and are left in cm->h_recv for the caller (e2s_pipeline_sharded).
// Everything the scan launches, enqueued on the context's stream without a synchronisation: accumulators zeroed, K1 + K2
// (k_lcp_flags + k_cluster_emit) or the one-pass k_cluster_scan + k_chunk_resolve.  s->last_one_pass says which.
static int scan_enqueue(e2s_shard* s, uint32_t k, int32_t min_len) {
    e2s_ctx* c = s->ctx;
    const char* env = getenv("E2S_CLUSTER_VARIANT");
    s->variant = env ? atoi(env) : 0;
    // One pass over the byte LCP (k_cluster_scan) whenever the shard has it and min_len allows the bit-parallel length
    // test; else the two-kernel path on the 4-byte LCP (k_lcp_flags + k_cluster_emit).  E2S_SCAN_LEGACY=1 forces the latter.
    const bool one_pass = s->last_one_pass = one_pass_ok(s, k, min_len) && !getenv("E2S_SCAN_LEGACY");
    const uint64_t num_tiles = emit_num_tiles(s->n_local);
    if (one_pass) {
        if (!s->d_chunks) {
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_chunks), SCAN_MAX_CHUNKS * sizeof(ChunkRec)) != cudaSuccess ||
                cudaMalloc(reinterpret_cast<void**>(&s->d_segs), SCAN_MAX_CHUNKS * sizeof(ChunkSeg)) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "chunk tables");
        }
        CU(c, scan_plan(s->n_local, c->sm_count, &s->n_chunks, &s->tiles_per_chunk));  // (n_local changes from chunk to chunk of a chunked shard)
        {
            const uint64_t want = (s->n_local / 8 + 4096) / s->n_chunks + 64;
            int rc = ensure_segments(s, want > s->seg_cap ? want : s->seg_cap);
            if (rc) return rc;
        }
    } else {
        if (!s->d_desc) {
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_desc), emit_desc_words() * 8) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "chunk descriptors");
            s->desc_cap = emit_desc_words();
        }
        if (!s->d_flags) {
            s->flag_words = flags_words_needed(s->n_local);
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_flags), s->flag_words * 2 * 4) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "flag masks");
            // K1 overwrites the words of its tiles; the tail up to K2's tile size stays zero
            CU(c, cudaMemsetAsync(s->d_flags, 0, s->flag_words * 2 * 4, c->stream));
        }
    }
    if (!one_pass && !s->d_start) {
        int rc = ensure_records(s, s->n_local / 8 + 4096);
        if (rc) return rc;
    }
    // K1: LCP -> START/END masks (two-kernel path only)
    if (!one_pass) {
        FlagParams fp;
        fp.lcp = s->lcp;
        fp.n_local = s->n_local;
        fp.global_off = s->global_off;
        fp.n_global = s->n_global;
        fp.k = k;
        fp.num_tiles = 0;
        fp.s_words = s->d_flags;
        fp.e_words = s->d_flags + s->flag_words;
        c->timer.begin(E2S_KERNEL_FLAGS, c->stream);
        cudaError_t le = launch_flags(fp, s->alloc_r / 32, c->sm_count, c->stream, s->variant);
        c->timer.end(c->stream);
        CU(c, le);
        ++c->launches;
    }
    CU(c, cudaMemsetAsync(s->d_res, 0, sizeof(ClusterDev), c->stream));
    if (!one_pass) CU(c, cudaMemsetAsync(s->d_desc, 0, s->desc_cap * 8, c->stream));
    EmitParams p;
    p.s_words = s->d_flags;
    p.e_words = s->d_flags + s->flag_words;
    p.num_tiles = num_tiles;
    p.global_off = s->global_off;
    p.n_global = s->n_global;
    p.min_len = min_len;
    p.out_start = s->d_start;
    p.out_len = s->d_len;
    p.cap = s->rec_cap - 4;  // room for adopted records
    p.desc = s->d_desc;
    p.planes = s->d_planes;
    p.pf_mcov = (s->pf_arm && s->sealed) ? s->pf_arm : 0;
    p.pf_list = nullptr;
    p.pf_cap = 0;
    if (p.pf_mcov) {
        uint64_t want = (one_pass ? s->seg_cap * s->n_chunks : s->rec_cap) / 16 + 4096;
        if (const char* dbg = getenv("E2S_PF_CAPACITY")) {  // test hook: a tiny list forces the overflow -> two-phase fallback
            const uint64_t v = strtoull(dbg, nullptr, 10);
            if (v) {
                want = v;
                if (s->pf_cap > v && !s->pf_want) s->pf_cap = v;  // also shrink the advertised capacity of an existing buffer
            }
        }
        if (s->pf_want > want) want = s->pf_want;  // (an overflow of the last attempt asked for more)
        if (want > s->pf_cap) {
            cudaFree(s->d_pf_list);
            s->d_pf_list = nullptr;
            s->pf_cap = 0;
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_pf_list), (want + 8) * sizeof(SurvEntry)) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "prefilter survivor list");
            s->pf_cap = want;
        }
        p.pf_list = s->d_pf_list;
        p.pf_cap = s->pf_cap > 4 ? s->pf_cap - 4 : 0;  // (room for the records k_merge_stats adopts)
    }
    p.dbg = nullptr;
    p.res = s->d_res;
    const bool is_last = s->global_off + s->n_local == s->n_global;
    p.tail_lcp = is_last ? s->lcp + s->n_local - 2 : nullptr;
    p.tail_bwt = is_last ? s->bwt + s->n_local - 1 : nullptr;
    if (one_pass) {
        CU(c, cudaMemsetAsync(s->d_chunks, 0, size_t(s->n_chunks) * sizeof(ChunkRec), c->stream));
        Scan8Params sp;
        sp.lcpt = s->lcpt;
        sp.planes = s->d_planes;
        sp.n_local = s->n_local;
        sp.global_off = s->global_off;
        sp.n_global = s->n_global;
        sp.k = k;
        sp.min_len = min_len;
        sp.num_tiles = 0;
        sp.n_chunks = s->n_chunks;
        sp.tiles_per_chunk = s->tiles_per_chunk;
        sp.seg_start = s->d_seg_start;
        sp.seg_len = s->d_seg_len;
        sp.seg_cap = s->seg_cap;
        sp.chunks = s->d_chunks;
        sp.pf_mcov = p.pf_mcov;
        sp.pf_list = p.pf_list;
        sp.pf_cap = p.pf_cap;
        sp.res = s->d_res;
        sp.tail_lcp = p.tail_lcp;
        sp.tail_bwt = p.tail_bwt;
        c->timer.begin(E2S_KERNEL_SCAN1, c->stream);
        cudaError_t le = launch_scan(sp, s->alloc_r, c->stream);
        c->timer.end(c->stream);
        CU(c, le);
        ResolveParams rp;
        rp.chunks = s->d_chunks;
        rp.segs = s->d_segs;
        rp.n_chunks = s->n_chunks;
        rp.min_len = min_len;
        rp.global_off = s->global_off;
        rp.n_global = s->n_global;
        rp.init_state = s->chunked ? s->carry_state : (s->global_off == 0 ? 0 : 1);
        rp.planes = s->d_planes;
        rp.pf_mcov = p.pf_mcov;
        rp.pf_list = p.pf_list;
        rp.pf_cap = p.pf_cap;
        rp.res = s->d_res;
        c->timer.begin(E2S_KERNEL_RESOLVE, c->stream);
        cudaError_t re = launch_chunk_resolve(rp, c->stream);
        c->timer.end(c->stream);
        CU(c, re);
        ++c->launches;
    } else {
        c->timer.begin(E2S_KERNEL_EMIT, c->stream);
        cudaError_t le = launch_emit(p, c->sm_count, c->stream);
        c->timer.end(c->stream);
        CU(c, le);
    }
    ++c->launches;
    return E2S_OK;
}

static int cluster_run_impl(e2s_shard* s, uint32_t k, int32_t min_len, e2s_cluster_summary* sum, e2s_comm* cm) {
    if (!s || !sum) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_cluster_run: NULL argument");
    e2s_ctx* c = s->ctx;
    if (s->chunked) return fail(c, E2S_ERR_STATE, "chunked shard: use e2s_chunk_begin / e2s_chunk_scan / e2s_chunked_finish");
    if (k == 0) return fail(c, E2S_ERR_ARG, "k must be >= 1 (the CLI maps 0 to the default 16)");
    CU(c, cudaSetDevice(c->device));
    if (!s->h_pin) CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_pin), sizeof(ClusterDev), cudaHostAllocDefault));
    ClusterDev& h = *s->h_pin;
    for (int attempt = 0; attempt < 2; ++attempt) {
        int erc = scan_enqueue(s, k, min_len);
        if (erc) return erc;
        const bool one_pass = s->last_one_pass;
        bool any_overflow = false;
        uint64_t max_written = 0;
        if (cm) {
            CU(c, launch_pack_exchange(s->d_res, s->n_local, s->global_off, uint64_t(s->lay_x), cm->d_send, c->stream));
            ++c->launches;
            if (int rc = all_gather_rows(c, cm)) return rc;
            CU(c, cudaMemcpyAsync(cm->h_recv, cm->d_recv, size_t(cm->world) * XR_WORDS * 8, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            memcpy(&h, cm->h_recv + size_t(cm->rank) * XR_WORDS, sizeof h);
            for (int g = 0; g < cm->world; ++g) {  // every rank sees every overflow flag: all of them repeat the round together
                const ClusterDev& hg = *reinterpret_cast<const ClusterDev*>(cm->h_recv + size_t(g) * XR_WORDS);
                any_overflow |= (hg.overflow & 1) != 0;  // (bit 1 = survivor list: not fatal here, find_events then runs its own prefilter)
                if (hg.n_written > max_written) max_written = hg.n_written;
            }
        } else {
            CU(c, cudaMemcpyAsync(&h, s->d_res, sizeof h, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            any_overflow = (h.overflow & 1) != 0;
            max_written = h.n_written;
        }
        if (!any_overflow) break;
        if (attempt == 1) return fail(c, E2S_ERR_STATE, "record buffer overflow after resize");
        if ((h.overflow & 1) || !cm) {
            const int rc = one_pass ? grow_segments(s) : ensure_records(s, (cm ? h.n_written : max_written) + 4096);
            if (rc) return rc;
        }
    }
    make_summary(h, s->n_local, s->global_off, s->n_global, k, min_len, uint64_t(s->lay_x), sum);
    s->h_res = h;
    s->pf_mcov = (s->pf_arm && s->sealed) ? s->pf_arm : 0;
    s->pf_count = h.n_pf;
    s->pf_ok = s->pf_mcov != 0 && !(h.overflow & 2) && h.n_pf + 4 <= s->pf_cap;
    s->pf_has_adopted = false;
    s->have_scan_stats = true;
    s->m_own = h.n_written;
    s->m_list = h.n_written;
    s->contiguous = !s->last_one_pass;
    s->have_clusters = true;
    s->staged = false;
    s->finalized = false;
    s->have_events = false;
    memset(&s->merged, 0, sizeof s->merged);
    return E2S_OK;
}



}  // extern "C"
// capacity of the payload / survivor list of a chunked shard (grown between chunks, contents kept)
template <typename T>
static cudaError_t grow_keep(T*& ptr, uint64_t& cap, uint64_t used, uint64_t need, cudaStream_t stream) {
    if (need <= cap && ptr) return cudaSuccess;
    const uint64_t ncap = need + need / 2 + 4096;
    T* np = nullptr;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&np), ncap * sizeof(T));
    if (e != cudaSuccess) return e;
    if (ptr && used) e = cudaMemcpyAsync(np, ptr, used * sizeof(T), cudaMemcpyDeviceToDevice, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    cudaFree(ptr);
    ptr = np;
    cap = ncap;
    return e;
}
extern "C" {

// copies the records of the survivors listed in d_pf_list[0, n) (base relative to the resident chunk) to the payload

static int capture_survivors(e2s_shard* s, uint64_t n, const unsigned long long* d_count = nullptr) {
    e2s_ctx* c = s->ctx;
    if (!n) return E2S_OK;
    const uint64_t need_pay = s->pay_used + n * uint64_t(MAX_C_LEN);
    uint64_t cap4 = s->pay_cap, cap1 = s->pay_cap, capt = s->pay_cap, caps = s->pay_cap;
    CU(c, grow_keep(s->p_lcp, cap4, s->pay_used, need_pay, c->stream));
    CU(c, grow_keep(s->p_text, capt, s->pay_used, need_pay, c->stream));
    CU(c, grow_keep(s->p_suff, caps, s->pay_used, need_pay, c->stream));
    CU(c, grow_keep(s->p_bwt, cap1, s->pay_used, need_pay, c->stream));
    s->pay_cap = cap4;
    CU(c, grow_keep(s->d_surv, s->surv_cap, s->surv_count, s->surv_count + n, c->stream));
    CaptureParams cp;
    cp.in = s->d_pf_list;
    cp.n_in = d_count ? d_count : &s->d_res->n_pf;
    cp.n_in_cap = n;
    cp.lcp = s->lcp;
    cp.text = s->text;
    cp.suff = s->suff;
    cp.bwt = s->bwt;
    cp.p_lcp = s->p_lcp;
    cp.p_text = s->p_text;
    cp.p_suff = s->p_suff;
    cp.p_bwt = s->p_bwt;
    cp.pay_cap = s->pay_cap;
    cp.out = s->d_surv;
    cp.out_cap = s->surv_cap;
    cp.counters = s->d_cap_counters;
    CU(c, launch_capture(cp, c->stream, c->sm_count));
    ++c->launches;
    unsigned long long hc[3] = {0, 0, 0};
    CU(c, cudaMemcpyAsync(hc, s->d_cap_counters, sizeof hc, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (hc[2] & 1)
        return fail(c, E2S_ERR_UNSUPPORTED,
                    "chunked shard: a cluster of 65 536 or more positions whose wrapped length passes the filters has left the device "
                    "(use a resident shard for this input)");
    if (hc[2]) return fail(c, E2S_ERR_STATE, "chunked shard: payload / survivor list capacity");
    const uint64_t pay0 = s->pay_used, surv0 = s->surv_count;
    s->pay_used = hc[0];
    s->surv_count = hc[1];
    if (s->host_gsa && hc[1] > surv0) {  // lean SoA mode: text / suff of the captured records come from the host's pairSA
        const uint64_t n_new = hc[1] - surv0, n_pay = hc[0] - pay0;
        if (n_new > s->h_surv_cap) {
            if (s->h_surv) cudaFreeHost(s->h_surv);
            s->h_surv = nullptr;
            s->h_surv_cap = 0;
            CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_surv), (n_new + n_new / 4 + 1024) * sizeof(SurvEntry), cudaHostAllocDefault));
            s->h_surv_cap = n_new + n_new / 4 + 1024;
        }
        if (2 * n_pay > s->h_gather_cap) {
            if (s->h_gather) cudaFreeHost(s->h_gather);
            s->h_gather = nullptr;
            s->h_gather_cap = 0;
            CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_gather), (2 * n_pay + n_pay / 2 + 4096) * 4, cudaHostAllocDefault));
            s->h_gather_cap = 2 * n_pay + n_pay / 2 + 4096;
        }
        CU(c, cudaMemcpyAsync(s->h_surv, s->d_surv + surv0, n_new * sizeof(SurvEntry), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        uint32_t* g_text = s->h_gather;
        uint32_t* g_suff = s->h_gather + n_pay;
        const uint64_t tail_lo = s->n_global > GSA_TAIL ? s->n_global - GSA_TAIL : 0;
        const int y = s->gsa_y, z = s->gsa_z, rs = y + z;
        auto le = [](const uint8_t* q, int nb) {
            uint32_t v = 0;
            for (int b = 0; b < (nb < 4 ? nb : 4); ++b) v |= uint32_t(q[b]) << (8 * b);
            return v;
        };
        bool any_tail = false;
        for (uint64_t i = 0; i < n_new; ++i) {
            const SurvEntry& e = s->h_surv[i];
            const uint64_t o = e.base - pay0;
            if (e.start >= tail_lo) {  // the device holds text / suff of these positions (and of the phantom records behind them)
                any_tail = true;
                continue;
            }
            const uint8_t* g = s->host_gsa + e.start * uint64_t(rs);  // suff(z) then text(y): ref:include.hpp:159-175
            // (an adopted record may run past the end of the eBWT: far longer than any analysed cluster, its records are never read)
            const uint64_t have = e.start + e.len <= s->n_global ? e.len : s->n_global - e.start;
            for (uint32_t j = 0; j < e.len; ++j, g += rs) {
                g_suff[o + j] = j < have ? le(g, z) : 0u;
                g_text[o + j] = j < have ? le(g + z, y) : 0u;
            }
        }
        if (any_tail) {  // their captured values come back first so that one copy can overwrite the whole range
            for (uint64_t i = 0; i < n_new; ++i) {
                const SurvEntry& e = s->h_surv[i];
                if (e.start < tail_lo) continue;
                CU(c, cudaMemcpyAsync(g_text + (e.base - pay0), s->p_text + e.base, size_t(e.len) * 4, cudaMemcpyDeviceToHost, c->stream));
                CU(c, cudaMemcpyAsync(g_suff + (e.base - pay0), s->p_suff + e.base, size_t(e.len) * 4, cudaMemcpyDeviceToHost, c->stream));
            }
            CU(c, cudaStreamSynchronize(c->stream));
        }
        CU(c, cudaMemcpyAsync(s->p_text + pay0, g_text, n_pay * 4, cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaMemcpyAsync(s->p_suff + pay0, g_suff, n_pay * 4, cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));  // (the staging is reused by the next chunk)
        s->lean_h2d += n_pay * 8;
        s->lean_d2h += n_new * sizeof(SurvEntry);
    }
    return E2S_OK;
}

// Scan of the chunk begun by e2s_chunk_begin, after its loads: seal, the one-pass scan with the state carried over from the
// chunks before, and -- mcov_out > 0: both tools will run -- the fused BWT prefilter with the survivors' records captured
// for phase 2.  *n_records = records of this chunk (e2s_cluster_fetch / _fetch_packed return exactly them until the next
// e2s_chunk_begin).
int e2s_chunk_scan(e2s_shard* s, uint32_t k, int32_t min_len, int mcov_out, uint64_t* n_records) {
    if (!s || !s->chunked || !s->chunk_open) return fail(s ? s->ctx : nullptr, E2S_ERR_STATE, "e2s_chunk_scan: begin a chunk first");
    e2s_ctx* c = s->ctx;
    if (k == 0) return fail(c, E2S_ERR_ARG, "k must be >= 1 (the CLI maps 0 to the default 16)");
    if (mcov_out < 0 || 2 * mcov_out > E2S_MAX_C_LEN) return fail(c, E2S_ERR_ARG, "e2s_chunk_scan: need 0 <= 2 * mcov_out <= 150");
    int rc = e2s_shard_seal(s);
    if (rc) return rc;
    if (!one_pass_ok(s, k, min_len))
        return fail(c, E2S_ERR_UNSUPPORTED,
                    "chunked shards need the one-pass scan: -m <= 33, and -k <= 127 when an LCP value exceeds 127; "
                    "use a resident shard for this input");
    if (!s->h_pin) CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_pin), sizeof(ClusterDev), cudaHostAllocDefault));
    ClusterDev& h = *s->h_pin;
    const uint32_t arm_before = s->pf_arm;
    s->pf_arm = uint32_t(mcov_out);
    for (int attempt = 0;; ++attempt) {
        if ((rc = scan_enqueue(s, k, min_len))) break;
        cudaError_t e = cudaMemcpyAsync(&h, s->d_res, sizeof h, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            rc = cuda_fail(c, e, "chunk scan");
            break;
        }
        if (!h.overflow) break;
        if (attempt >= 2) {
            rc = fail(c, E2S_ERR_STATE, "record / survivor buffers still too small after two resizes");
            break;
        }
        if ((h.overflow & 1) && (rc = grow_segments(s))) break;
        if (h.overflow & 2) s->pf_want = h.n_pf + h.n_pf / 8 + 4096;
    }
    s->pf_arm = arm_before;
    if (rc) return rc;
    if (mcov_out && h.n_pf && (rc = capture_survivors(s, h.n_pf))) return rc;
    // the range's accumulators; the state the next chunk starts from
    ClusterDev& a = s->acc;
    a.n_end += h.n_end;
    a.n_written += h.n_written;
    if (!a.head_end) a.head_end = h.head_end;
    a.any_event |= h.any_event;
    a.open_start = h.open_start;
    if (h.end_nm2_start) a.end_nm2_start = h.end_nm2_start;
    if (h.n_written) a.last_rec = h.last_rec;
    a.n_bases += h.n_bases;
    for (int i = 0; i < E2S_HIST_BINS; ++i) a.hist[i] += h.hist[i];
    if (s->global_off + s->n_local == s->n_global) {
        a.tail_lcp_nm2 = h.tail_lcp_nm2;
        a.tail_lcp_nm1 = h.tail_lcp_nm1;
        a.tail_bwt_nm1 = h.tail_bwt_nm1;
    }
    a.ticket++;  // chunks scanned
    if (a.any_event) s->carry_state = h.open_start ? h.open_start - 1 + 2 : 0;
    s->chunk_open = false;
    s->h_res = h;
    s->pf_mcov = uint32_t(mcov_out);
    s->m_own = s->m_list = h.n_written;
    s->contiguous = false;
    s->have_clusters = true;
    s->staged = false;
    s->finalized = false;
    s->have_events = false;
    s->have_scan_stats = true;
    memset(&s->merged, 0, sizeof s->merged);
    if (n_records) *n_records = h.n_written;
    return E2S_OK;
}

// clust2snp on a chunked shard (an index larger than device memory): instead of scanning the chunk for clusters, take them from
// the .clusters file -- the m records whose START lies in the open chunk, 10 bytes each, in file order -- run the BWT prefilter of
// find_variants on them (K3a, ref:clust2snp.cpp:402-429) and keep the EGSA records of the survivors for phase 2.
// max_clust_length comes from statistics() over the whole file (ref:clust2snp.cpp:877-966), which needs no index.
int e2s_chunk_stage_clusters(e2s_shard* s, const void* rec10, uint64_t m, int mcov_out, int max_clust_length, uint64_t* n_survivors) {
    if (!s || !s->chunked || !s->chunk_open) return fail(s ? s->ctx : nullptr, E2S_ERR_STATE, "e2s_chunk_stage_clusters: begin a chunk first");
    e2s_ctx* c = s->ctx;
    if (m && !rec10) return fail(c, E2S_ERR_ARG, "e2s_chunk_stage_clusters: NULL records");
    if (mcov_out < 1 || 2 * mcov_out > E2S_MAX_C_LEN || max_clust_length > E2S_MAX_C_LEN)
        return fail(c, E2S_ERR_UNSUPPORTED, "e2s_chunk_stage_clusters: need 2 <= 2 * mcov_out <= 150 and max_clust_length <= 150");
    if (s->acc.ticket && s->pf_mcov != uint32_t(mcov_out)) return fail(c, E2S_ERR_ARG, "e2s_chunk_stage_clusters: one -m for all the chunks of a range");
    int rc = e2s_shard_seal(s);
    if (rc) return rc;
    if (n_survivors) *n_survivors = 0;
    if (m) {
        if ((rc = ensure_records(s, m + 8))) return rc;
        std::vector<uint64_t> st(m);
        std::vector<uint16_t> ln(m);
        const uint8_t* r = static_cast<const uint8_t*>(rec10);
        for (uint64_t i = 0; i < m; ++i) {
            get_rec10(r + i * 10, &st[i], &ln[i]);
            if (st[i] - s->global_off >= s->n_local) return fail(c, E2S_ERR_ARG, "e2s_chunk_stage_clusters: a record does not start in the open chunk");
            if (ln[i] <= E2S_MAX_C_LEN) s->acc.hist[ln[i]]++;
        }
        if (m + 8 > s->pf_cap) {  // every record may survive
            cudaFree(s->d_pf_list);
            s->d_pf_list = nullptr;
            s->pf_cap = 0;
            const uint64_t want = m + m / 4 + 4096;
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_pf_list), (want + 8) * sizeof(SurvEntry)) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "survivor list");
            s->pf_cap = want;
        }
        if (!s->d_stage_dev) CU(c, cudaMalloc(reinterpret_cast<void**>(&s->d_stage_dev), sizeof(SnpDev)));
        CU(c, cudaMemsetAsync(s->d_stage_dev, 0, sizeof(SnpDev), c->stream));
        CU(c, cudaMemcpyAsync(s->d_start, st.data(), m * 8, cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaMemcpyAsync(s->d_len, ln.data(), m * 2, cudaMemcpyHostToDevice, c->stream));
        SnpArrays a = shard_arrays(s);
        a.cl_start = s->d_start;
        a.cl_len = s->d_len;
        a.m = m;
        CU(c, launch_code_scan(a, uint32_t(mcov_out), uint32_t(max_clust_length), s->d_pf_list, s->pf_cap, s->d_stage_dev, c->stream, c->sm_count));
        ++c->launches;
        SnpDev h;
        CU(c, cudaMemcpyAsync(&h, s->d_stage_dev, sizeof h, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));  // (also: st / ln leave this frame)
        if (h.n_survivors && (rc = capture_survivors(s, h.n_survivors, &s->d_stage_dev->n_survivors))) return rc;
        if (n_survivors) *n_survivors = h.n_survivors;
    }
    s->acc.ticket++;  // chunks done
    s->acc.n_written += m;
    s->chunk_open = false;
    s->pf_mcov = uint32_t(mcov_out);
    return E2S_OK;
}

// After the last chunk of the range went through e2s_chunk_stage_clusters: e2s_find_events runs on the captured records.
int e2s_chunked_clusters_finish(e2s_shard* s) {
    if (!s || !s->chunked) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunked_clusters_finish: not a chunked shard");
    e2s_ctx* c = s->ctx;
    if (s->chunk_open || s->global_off + s->n_local != s->range_lo + s->range_n || !s->acc.ticket)
        return fail(c, E2S_ERR_STATE, "e2s_chunked_clusters_finish: the last chunk of the range has not been staged");
    s->h_res = s->acc;  // (the length histogram of the staged records: n_analysed of e2s_find_events)
    s->m_own = s->m_list = s->acc.n_written;
    s->records_flushed = true;
    s->have_clusters = true;
    s->staged = false;
    s->finalized = true;
    s->have_events = false;
    s->have_scan_stats = false;
    s->pf_ok = true;
    s->pf_has_adopted = true;
    memset(&s->merged, 0, sizeof s->merged);
    return E2S_OK;
}

// After the last chunk: the summary of the shard's whole range, as e2s_cluster_run returns it for a resident shard.  From
// here on e2s_cluster_merge / e2s_cluster_finalize / e2s_statistics / e2s_find_events work as usual (the records themselves
// were handed out chunk by chunk; phase 2 runs on the captured survivors).
int e2s_chunked_finish(e2s_shard* s, uint32_t k, int32_t min_len, e2s_cluster_summary* sum) {
    if (!s || !s->chunked || !sum) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunked_finish: not a chunked shard");
    e2s_ctx* c = s->ctx;
    if (s->chunk_open || s->global_off + s->n_local != s->range_lo + s->range_n || !s->acc.ticket)
        return fail(c, E2S_ERR_STATE, "e2s_chunked_finish: the last chunk of the range has not been scanned");
    const ClusterDev& h = s->acc;
    make_summary(h, s->range_n, s->range_lo, s->n_global, k, min_len, uint64_t(s->lay_x), sum);
    s->h_res = h;  // statistics() of the whole range
    s->m_own = s->m_list = h.n_written;
    s->records_flushed = true;
    s->pf_ok = s->pf_mcov != 0;
    s->pf_has_adopted = false;
    return E2S_OK;
}

int e2s_cluster_run(e2s_shard* s, uint32_t k, int32_t min_len, e2s_cluster_summary* sum) {
    return cluster_run_impl(s, k, min_len, sum, nullptr);
}

// Host-only: chain the shards' open-cluster states, resolve head records, apply the tail rule with
// the post-EOF phantom record (ref:ebwt2clust.cpp:90-135; SURVEY.md §8(a) A3).
static const char* merge_message(int rc) {
    switch (rc) {
        case MERGE_NOT_PARTITION: return "e2s_cluster_merge: shards are not a partition of [0, n_global)";
        case MERGE_NOT_COVER: return "e2s_cluster_merge: shards do not cover n_global";
        case MERGE_END_WITHOUT_START: return "e2s_cluster_merge: END without START (inconsistent summaries)";
        case MERGE_EMPTY: return "empty .clusters (the reference divides by zero here)";
        case MERGE_BAD_MCOV: return "2*mcov_out outside [0,150]";
        default: return "merge failed";
    }
}
static int merge_status(int rc) {
    return rc == MERGE_END_WITHOUT_START ? E2S_ERR_STATE : ((rc == MERGE_EMPTY || rc == MERGE_BAD_MCOV) ? E2S_ERR_UNSUPPORTED : E2S_ERR_ARG);
}

int e2s_cluster_merge(const e2s_cluster_summary* all, int n_shards, int my, e2s_cluster_merged* out) {
    if (!all || !out || n_shards < 1 || my < 0 || my >= n_shards) return fail(nullptr, E2S_ERR_ARG, "e2s_cluster_merge: bad argument");
    const int rc = merge_core(all, n_shards, my, out);  // merge.cuh: the same code k_merge_stats runs on the device
    if (rc != MERGE_OK) return fail(nullptr, merge_status(rc), merge_message(rc));
    return E2S_OK;
}

int e2s_cluster_finalize(e2s_shard* s, const e2s_cluster_merged* mg) {
    if (!s || !mg) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_cluster_finalize: NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->have_clusters || s->staged) return fail(c, E2S_ERR_STATE, "e2s_cluster_finalize: run e2s_cluster_run first");
    CU(c, cudaSetDevice(c->device));
    s->merged = *mg;
    s->m_list = s->m_own + mg->n_adopt;  // the adopted records join the device list when a pass over it needs them (find_events)
    s->adopt_put = false;
    s->finalized = true;
    if (s->chunked && s->pf_mcov && mg->n_adopt) {  // their records are still on the device (the range's last chunk): to the payload
        // only the lengths phase 2 analyses (2 mcov_out .. 150): any other adopted record is never read, and may be far longer
        // than the payload reserves per record or start in a chunk that has left the device
        SurvEntry extra[4];
        unsigned long long n = 0;
        for (uint32_t i = 0; i < mg->n_adopt && i < 4; ++i)
            if (mg->adopt_len[i] >= 2 * uint64_t(s->pf_mcov) && mg->adopt_len[i] <= uint64_t(E2S_MAX_C_LEN))
                extra[n++] = SurvEntry{mg->adopt_start[i], mg->adopt_start[i] - s->global_off, uint32_t(mg->adopt_len[i]), 0u};
        if (n) {
            CU(c, cudaMemcpyAsync(s->d_pf_list, extra, n * sizeof(SurvEntry), cudaMemcpyHostToDevice, c->stream));
            CU(c, cudaMemcpyAsync(&s->d_res->n_pf, &n, 8, cudaMemcpyHostToDevice, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            int rc = capture_survivors(s, n);
            if (rc) return rc;
        }
        s->pf_has_adopted = true;
    }
    return E2S_OK;
}

int e2s_cluster_lm(e2s_shard* s, uint32_t k, int32_t min_len, uint64_t* n_written, uint64_t* n_clust_out) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (s->global_off != 0 || s->n_local != s->n_global)
        return fail(s->ctx, E2S_ERR_ARG, "e2s_cluster_lm needs the whole eBWT in one shard; use run + merge + finalize");
    e2s_cluster_summary sum;
    int rc = e2s_cluster_run(s, k, min_len, &sum);
    if (rc) return rc;
    e2s_cluster_merged mg;
    rc = e2s_cluster_merge(&sum, 1, 0, &mg);
    if (rc) {
        s->ctx->err = g_err;
        return rc;
    }
    rc = e2s_cluster_finalize(s, &mg);
    if (rc) return rc;
    if (n_written) *n_written = mg.total_written;
    if (n_clust_out) *n_clust_out = mg.n_clust_out;
    return E2S_OK;
}

// records of this shard in .clusters order: [head] + own + [tail]
static uint64_t out_count(const e2s_shard* s) {
    if (s->staged) return s->m_own;
    return s->m_own + (s->merged.n_prepend && s->merged.prepend_written ? 1 : 0) + s->merged.n_append;
}

int e2s_cluster_count(const e2s_shard* s, uint64_t* m) {
    if (!s || !m) return fail(nullptr, E2S_ERR_ARG, "NULL argument");
    if (!s->have_clusters) return fail(s->ctx, E2S_ERR_STATE, "no clusters yet");
    *m = out_count(s);
    return E2S_OK;
}

int e2s_cluster_fetch(e2s_shard* s, uint64_t* start, uint16_t* len, uint64_t cap, uint64_t* m) {
    if (!s || !start || !len || !m) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->have_clusters) return fail(c, E2S_ERR_STATE, "no clusters yet");
    if (s->records_flushed) return fail(c, E2S_ERR_STATE, "chunked shard: the records were handed out chunk by chunk");
    const uint64_t total = out_count(s);
    *m = total;
    if (cap < total) return fail(c, E2S_ERR_ARG, "e2s_cluster_fetch: capacity too small");
    CU(c, cudaSetDevice(c->device));
    uint64_t o = 0;
    if (!s->staged && s->merged.n_prepend && s->merged.prepend_written) {
        start[o] = s->merged.prepend_start;
        len[o] = uint16_t(s->merged.prepend_len);
        ++o;
    }
    if (s->m_own) {
        int rc = ensure_contiguous(s);
        if (rc) return rc;
        CU(c, cudaMemcpyAsync(start + o, s->d_start, s->m_own * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(len + o, s->d_len, s->m_own * 2, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        o += s->m_own;
    }
    if (!s->staged)
        for (uint32_t i = 0; i < s->merged.n_append; ++i) {
            start[o] = s->merged.append_start[i];
            len[o] = uint16_t(s->merged.append_len[i]);
            ++o;
        }
    return E2S_OK;
}

int e2s_cluster_fetch_packed(e2s_shard* s, void* rec10, uint64_t cap, uint64_t* m) {
    if (!s || !rec10 || !m) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->have_clusters) return fail(c, E2S_ERR_STATE, "no clusters yet");
    if (s->records_flushed) return fail(c, E2S_ERR_STATE, "chunked shard: the records were handed out chunk by chunk");
    const uint64_t total = out_count(s);
    *m = total;
    if (cap < total) return fail(c, E2S_ERR_ARG, "e2s_cluster_fetch_packed: capacity too small");
    CU(c, cudaSetDevice(c->device));
    uint8_t* o = static_cast<uint8_t*>(rec10);
    auto put = [&](uint64_t st, uint64_t ln) {
        put_rec10(o, st, ln);
        o += 10;
    };
    if (!s->staged && s->merged.n_prepend && s->merged.prepend_written) put(s->merged.prepend_start, s->merged.prepend_len);
    if (s->m_own) {  // pack on the device, one D2H straight into the caller's buffer
        if (s->m_own > s->packed_cap) {
            cudaFree(s->d_packed);
            s->d_packed = nullptr;
            s->packed_cap = 0;
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_packed), s->m_own * 10 + 16) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "packed record buffer");
            s->packed_cap = s->m_own;
        }
        if (s->contiguous)
            CU(c, launch_pack_records(s->d_start, s->d_len, s->m_own, s->d_packed, c->stream, c->sm_count));
        else  // straight from the scan's segments
            CU(c, launch_export_records(s->d_segs, s->n_chunks, s->seg_cap, s->d_seg_start, s->d_seg_len, nullptr, nullptr, s->d_packed, c->stream));
        ++c->launches;
        CU(c, cudaMemcpyAsync(o, s->d_packed, s->m_own * 10, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        o += s->m_own * 10;
    }
    if (!s->staged)
        for (uint32_t i = 0; i < s->merged.n_append; ++i) put(s->merged.append_start[i], s->merged.append_len[i]);
    return E2S_OK;
}

// ---------------------------------------------------------------------------------------------
// phase 2
// ---------------------------------------------------------------------------------------------
int e2s_clusters_stage(e2s_shard* s, const uint64_t* start, const uint16_t* len, uint64_t m) {
    if (!s || (m && (!start || !len))) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    int rc = ensure_records(s, m + 8);
    if (rc) return rc;
    if (m) {
        CU(c, cudaMemcpyAsync(s->d_start, start, m * 8, cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaMemcpyAsync(s->d_len, len, m * 2, cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    s->m_own = s->m_list = m;
    s->contiguous = true;
    s->pf_ok = false;
    s->have_clusters = true;
    s->staged = true;
    s->have_scan_stats = false;
    s->finalized = true;
    s->have_events = false;
    memset(&s->merged, 0, sizeof s->merged);
    return E2S_OK;
}

int e2s_clusters_stage_packed(e2s_shard* s, const void* rec10, uint64_t m) {
    if (!s || (m && !rec10)) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    std::vector<uint64_t> st(m);
    std::vector<uint16_t> ln(m);
    const uint8_t* r = static_cast<const uint8_t*>(rec10);
    for (uint64_t i = 0; i < m; ++i) get_rec10(r + i * 10, &st[i], &ln[i]);
    return e2s_clusters_stage(s, st.data(), ln.data(), m);
}

int e2s_statistics(e2s_shard* s, e2s_stats* st) {
    if (!s || !st) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->have_clusters) return fail(c, E2S_ERR_STATE, "no clusters yet");
    CU(c, cudaSetDevice(c->device));
    memset(st, 0, sizeof *st);
    if (!s->staged && s->have_scan_stats) {  // the scan accumulated the histogram of its own records
        for (int i = 0; i < E2S_HIST_BINS; ++i) st->hist[i] = s->h_res.hist[i];
        st->n_bases = s->h_res.n_bases;
        st->n_clust = s->m_own;
        st->last_len = s->h_res.last_rec & 0xffff;
    } else {
    unsigned long long h[E2S_HIST_BINS + 1];
    CU(c, cudaMemsetAsync(s->d_hist, 0, sizeof h, c->stream));
    CU(c, launch_len_hist(s->d_len, s->m_own, s->d_hist, c->stream, c->sm_count));
    ++c->launches;
    CU(c, cudaMemcpyAsync(h, s->d_hist, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    uint16_t last = 0;
    if (s->m_own) CU(c, cudaMemcpyAsync(&last, s->d_len + s->m_own - 1, 2, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < E2S_HIST_BINS; ++i) st->hist[i] = h[i];
    st->n_bases = h[E2S_HIST_BINS];
    st->n_clust = s->m_own;
    st->last_len = last;
    }
    auto add = [&](uint64_t l) {
        if (l <= E2S_MAX_C_LEN) st->hist[l]++;
        st->n_bases += l;
        st->n_clust++;
        st->last_len = l;
    };
    if (!s->staged) {
        if (s->merged.n_prepend && s->merged.prepend_written) {
            const uint64_t keep_last = st->last_len;
            add(s->merged.prepend_len);
            if (s->m_own) st->last_len = keep_last;  // the head record comes first, not last
        }
        for (uint32_t i = 0; i < s->merged.n_append; ++i) add(s->merged.append_len[i]);
    }
    return E2S_OK;
}

// ref:clust2snp.cpp:889-946: the last record is counted twice; then the pval loop
int e2s_statistics_finish(e2s_stats* st, uint64_t last_len, int mcov_out, double pval) {
    if (!st) return fail(nullptr, E2S_ERR_ARG, "NULL argument");
    const int rc = stats_finish_core(st, last_len, mcov_out, pval);  // merge.cuh
    if (rc != MERGE_OK) return fail(nullptr, merge_status(rc), merge_message(rc));
    return E2S_OK;
}

// Host-only: what every rank does with the all-gathered (summary, own-record statistics) rows between the phases.
int e2s_exchange_finish(const e2s_cluster_summary* sums, const e2s_stats* own, int n_shards, int my, int mcov_out, double pval,
                        e2s_cluster_merged* mine, e2s_stats* total) {
    if (!sums || !own || !mine || !total || n_shards < 1 || my < 0 || my >= n_shards)
        return fail(nullptr, E2S_ERR_ARG, "e2s_exchange_finish: bad argument");
    memset(total, 0, sizeof *total);
    uint64_t last_len = 0;
    bool any = false;
    for (int g = 0; g < n_shards; ++g) {
        e2s_cluster_merged mg;
        int rc = e2s_cluster_merge(sums, n_shards, g, &mg);
        if (rc) return rc;
        if (g == my) *mine = mg;
        // records of shard g in file order: [head record] own records [tail records]
        e2s_stats st = own[g];
        auto add = [&](uint64_t l, bool is_last) {
            if (l <= E2S_MAX_C_LEN) st.hist[l]++;
            st.n_bases += l;
            st.n_clust++;
            if (is_last) st.last_len = l;
        };
        if (mg.n_prepend && mg.prepend_written) add(mg.prepend_len, own[g].n_clust == 0);
        for (uint32_t i = 0; i < mg.n_append; ++i) add(mg.append_len[i], true);
        for (int i = 0; i < E2S_HIST_BINS; ++i) total->hist[i] += st.hist[i];
        total->n_clust += st.n_clust;
        total->n_bases += st.n_bases;
        if (st.n_clust) {
            last_len = st.last_len;
            any = true;
        }
    }
    total->last_len = last_len;
    if (!any) return fail(nullptr, E2S_ERR_UNSUPPORTED, "empty .clusters (the reference divides by zero here)");
    return e2s_statistics_finish(total, last_len, mcov_out, pval);
}

void e2s_snp_default_params(e2s_snp_params* p) {
    memset(p, 0, sizeof *p);
    p->k_left = 31;
    p->k_right = 30;
    p->mcov_out = 5;
    p->max_gap = 10;
    p->consensus_reads = 20;
    p->max_err = 2;
    p->max_snvs = 3;
    p->pval = 0.99;
}

static bool snp_params_ok(const e2s_snp_params* p) {
    return !(p->k_left < 1 || p->k_left > E2S_MAX_K || p->k_right < 1 || p->k_right > E2S_MAX_K || p->max_gap < 1 ||
             p->max_gap > p->k_left || p->max_gap > 255 || p->mcov_out < 1 || 2 * p->mcov_out > E2S_MAX_C_LEN || p->consensus_reads < 1);
}

int e2s_find_events(e2s_shard* s, const e2s_snp_params* p, int max_clust_length, e2s_snp_counts* counts) {
    if (!s || !p || !counts) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->have_clusters || !s->finalized) return fail(c, E2S_ERR_STATE, "clusters not computed / staged yet");
    if (!s->sealed) return fail(c, E2S_ERR_STATE, "call e2s_shard_seal after loading the shard");
    if (!c->d_bases) return fail(c, E2S_ERR_STATE, "stage the reads first (e2s_reads_stage)");
    if (!snp_params_ok(p) || max_clust_length > E2S_MAX_C_LEN)
        return fail(c, E2S_ERR_UNSUPPORTED, "clust2snp parameters outside the supported range (DESIGN.md)");
    CU(c, cudaSetDevice(c->device));
    s->have_events = false;
    s->events.clear();
    if (s->staged && s->m_list > 1) {
        // the reference assumes position-ordered, disjoint records (ref:clust2snp.cpp:818-833)
        SnpDev* chk = nullptr;
        CU(c, cudaMalloc(reinterpret_cast<void**>(&chk), sizeof(SnpDev)));
        cudaMemsetAsync(chk, 0, sizeof(SnpDev), c->stream);
        launch_check_sorted(s->d_start, s->d_len, s->m_list, chk, c->stream, c->sm_count);
        ++c->launches;
        SnpDev h;
        cudaMemcpyAsync(&h, chk, sizeof h, cudaMemcpyDeviceToHost, c->stream);
        cudaError_t e = cudaStreamSynchronize(c->stream);
        cudaFree(chk);
        if (e != cudaSuccess) return cuda_fail(c, e, "check_sorted");
        if (h.unsorted) return fail(c, E2S_ERR_UNSUPPORTED, ".clusters records are not position-ordered and disjoint");
    }
    SnpArrays a = shard_arrays(s);
    // K2 already ran the BWT prefilter for this -m (fused mode): its survivors + the records adopted from the merge
    // (which K2 did not see) replace K3a
    const SurvEntry* pre_list = nullptr;
    uint64_t pre_count = 0;
    if (s->chunked) {
        // the range went through the device chunk by chunk: phase 2 runs on the records e2s_chunk_scan captured for the
        // clusters that survived its prefilter
        if (!s->records_flushed || !s->pf_ok || s->pf_mcov != uint32_t(p->mcov_out))
            return fail(c, E2S_ERR_STATE, "chunked shard: phase 2 needs e2s_chunk_scan(mcov_out = this -m) on every chunk and e2s_chunked_finish");
        a.lcp = s->p_lcp;
        a.text = s->p_text;
        a.suff = s->p_suff;
        a.bwt = s->p_bwt;
        a.planes = nullptr;
        pre_list = s->d_surv;
        pre_count = s->surv_count;
        if (!pre_count) {  // nothing survived: no candidates
            memset(counts, 0, sizeof *counts);
            uint64_t na0 = 0;
            for (int l = 2 * p->mcov_out; l <= max_clust_length; ++l) na0 += s->h_res.hist[l];
            counts->n_analysed = na0;
            s->n_variants = 0;
            s->events_expanded = false;
            s->have_events = true;
            return E2S_OK;
        }
    } else if (!s->staged && s->pf_ok && s->pf_mcov == uint32_t(p->mcov_out) && max_clust_length <= E2S_MAX_C_LEN) {
        SurvEntry extra[4];
        const uint64_t n_extra = s->pf_has_adopted ? 0 : s->merged.n_adopt;  // <= 3 records the merge created and this shard analyses
        for (uint64_t i = 0; i < n_extra && i < 4; ++i)
            extra[i] = SurvEntry{s->merged.adopt_start[i], s->merged.adopt_start[i] - s->global_off, uint32_t(s->merged.adopt_len[i]), 0u};
        if (n_extra) {
            CU(c, cudaMemcpyAsync(s->d_pf_list + s->pf_count, extra, n_extra * sizeof(SurvEntry), cudaMemcpyHostToDevice, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));  // (extra[] lives on this stack frame)
        }
        s->pf_has_adopted = true;
        s->pf_count += n_extra;
        pre_list = s->d_pf_list;
        pre_count = s->pf_count;
    } else {
        int rc = ensure_contiguous(s);  // the two-phase path walks the record list: own records, then the adopted ones
        if (rc) return rc;
        if (!s->staged && s->merged.n_adopt && !s->adopt_put) {
            CU(c, launch_put_records(s->d_start, s->d_len, s->m_own, s->merged.adopt_start, s->merged.adopt_len, int(s->merged.n_adopt), c->stream));
            ++c->launches;
            s->adopt_put = true;
        }
    }
    a.cl_start = s->d_start;
    a.cl_len = s->d_len;
    a.m = s->m_list;
    const char* err = "";
    cudaError_t e = snp_run(s->work, a, *p, max_clust_length, c->d_bases, c->d_off, c->n_reads, c->sm_count, c->stream,
                            counts, &c->launches, &err, &c->timer, pre_list, pre_count);
    if (pre_list && e == cudaSuccess) counts->n_analysed = analysed_count(s->h_res, s->merged, p->mcov_out, max_clust_length);
    if (e == cudaErrorInvalidValue && err && strstr(err, "outside the staged reads")) return fail(c, E2S_ERR_UNSUPPORTED, err);
    if (e != cudaSuccess) return cuda_fail(c, e, err);
    // the packed candidates are already in pinned host memory (K4 wrote them there); they are expanded
    // into e2s_event records when e2s_events_fetch asks for them
    s->n_variants = counts->n_variants;
    s->events_expanded = false;
    s->have_events = true;
    return E2S_OK;
}

int e2s_events_fetch(e2s_shard* s, e2s_event* events, uint64_t cap, uint64_t* n) {
    if (!s || !n) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    if (!s->have_events) return fail(s->ctx, E2S_ERR_STATE, "run e2s_find_events first");
    *n = s->n_variants;
    if (!events) return E2S_OK;
    if (!s->events_expanded) {
        uint64_t nv = 0;
        s->events.resize(s->n_variants);
        cudaError_t e = snp_fetch_events(s->work, s->events.data(), s->n_variants, &nv, s->ctx->stream);
        if (e != cudaSuccess) return cuda_fail(s->ctx, e, "snp_fetch_events");
        if (nv != s->n_variants) return fail(s->ctx, E2S_ERR_STATE, "event count mismatch between device counter and packed records");
        s->events_expanded = true;
    }
    if (!events) return E2S_OK;
    if (cap < s->events.size()) return fail(s->ctx, E2S_ERR_ARG, "e2s_events_fetch: capacity too small");
    if (!s->events.empty()) memcpy(events, s->events.data(), s->events.size() * sizeof(e2s_event));
    return E2S_OK;
}

// to_file(): ref:clust2snp.cpp:633-780
int e2s_events_format(const e2s_event* ev, uint64_t n, uint64_t first_id, const e2s_snp_params* p, char** text, size_t* len) {
    if ((!ev && n) || !p || !text || !len) return fail(nullptr, E2S_ERR_ARG, "NULL argument");
    std::string out;
    out.reserve(size_t(n) * 200);
    uint64_t id = first_id;
    const int kl = p->k_left;
    for (uint64_t i = 0; i < n; ++i) {
        const e2s_event& e = ev[i];
        if (!e.keep) continue;
        std::string type;
        if (e.gap == 0) {
            type += e.left0[kl - 1];
            type += '/';
            type += e.left1[kl - 1];
        } else if (e.gap > 0) {
            type.append(e.left0 + kl - e.gap, size_t(e.gap));
            type += '/';
        } else {
            type += '/';
            type.append(e.left1 + kl + e.gap, size_t(-e.gap));
        }
        for (int path = 0; path < 2; ++path) {
            out += e.gap != 0 ? (path ? ">INDEL_lower_path_" : ">INDEL_higher_path_") : (path ? ">SNP_lower_path_" : ">SNP_higher_path_");
            out += std::to_string(id);
            out += "|P_1:";
            out += std::to_string(e.right_len);
            out += "_";
            out += type;
            out += "|";
            out += std::to_string(path ? e.supp1 : e.supp0);
            out += "|nb_pol_1\n";
            int skip = 0;
            if (path == 0 && e.gap < 0) skip = -e.gap;
            if (path == 1 && e.gap > 0) skip = e.gap;
            out.append((path ? e.left1 : e.left0) + skip, size_t(kl - skip));
            out.append(e.right, size_t(e.right_len));
            out += '\n';
        }
        ++id;
    }
    char* buf = static_cast<char*>(malloc(out.size() + 1));
    if (!buf) return fail(nullptr, E2S_ERR_NOMEM, "malloc");
    memcpy(buf, out.data(), out.size());
    buf[out.size()] = 0;
    *text = buf;
    *len = out.size();
    return E2S_OK;
}

void e2s_free(void* p) { free(p); }

// ---------------------------------------------------------------------------------------------
// end to end over host buffers
// ---------------------------------------------------------------------------------------------
// ebwt2clust + clust2snp on a sealed shard that holds the whole eBWT (one GPU), reads already staged
// Both phases on a sealed resident shard without leaving the stream in between: scan (+ the shard's exchange row, all-
// gathered by NCCL when there is a communicator) -> k_merge_stats (merge of all shards, tail / phantom rule, statistics(),
// max_clust_length: device memory) -> K3x / K3b / K4 on the scan's survivor list -> ONE copy of the results, ONE
// synchronisation.  Needs the fused prefilter (valid -m); the caller falls back to the host-driven sequence otherwise.
static int pipeline_step(e2s_shard* s, e2s_comm* cm, uint32_t k, int32_t min_len, const e2s_snp_params* p, e2s_cluster_merged* mg_out,
                         e2s_stats* st_out, e2s_snp_counts* cnt_out) {
    e2s_ctx* c = s->ctx;
    if (k == 0) return fail(c, E2S_ERR_ARG, "k must be >= 1 (the CLI maps 0 to the default 16)");
    if (!s->sealed) return fail(c, E2S_ERR_STATE, "call e2s_shard_seal after loading the shard");
    if (!c->d_bases) return fail(c, E2S_ERR_STATE, "stage the reads first (e2s_reads_stage)");
    if (!snp_params_ok(p)) return fail(c, E2S_ERR_UNSUPPORTED, "clust2snp parameters outside the supported range (DESIGN.md)");
    CU(c, cudaSetDevice(c->device));
    const int world = cm ? cm->world : 1, my = cm ? cm->rank : 0;
    if (world > MERGE_MAX_SHARDS) return fail(c, E2S_ERR_UNSUPPORTED, "more shards than k_merge_stats handles");
    if (!s->d_mout) {
        CU(c, cudaMalloc(reinterpret_cast<void**>(&s->d_mout), sizeof(MergeOut)));
        CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_mout), sizeof(MergeOut), cudaHostAllocDefault));
        CU(c, cudaMalloc(reinterpret_cast<void**>(&s->d_row), XR_WORDS * 8));
    }
    if (!s->h_pin) CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_pin), sizeof(ClusterDev), cudaHostAllocDefault));
    ClusterDev& h = *s->h_pin;
    MergeOut& mo = *s->h_mout;
    const uint32_t arm_before = s->pf_arm;
    s->pf_arm = uint32_t(p->mcov_out);
    s->have_events = false;
    s->events.clear();
    const SnpArrays a = shard_arrays(s);  // (phase 2 starts from the survivor list: the record list is not walked)
    const char* err = "";
    int rc = E2S_OK;
    for (int attempt = 0;; ++attempt) {
        if ((rc = scan_enqueue(s, k, min_len))) break;
        uint64_t* send = cm ? cm->d_send : s->d_row;
        const uint64_t* rows = send;
        c->timer.begin(E2S_KERNEL_MERGE, c->stream);
        if ((rc = launch_pack_exchange(s->d_res, s->n_local, s->global_off, uint64_t(s->lay_x), send, c->stream) == cudaSuccess ? 0 : 1)) {
            c->timer.end(c->stream);
            rc = fail(c, E2S_ERR_CUDA, "k_pack_exchange");
            break;
        }
        if (cm) {
            if ((rc = all_gather_rows(c, cm))) {
                c->timer.end(c->stream);
                break;
            }
            rows = cm->d_recv;
        }
        MergeParams mp;
        mp.rows = reinterpret_cast<const unsigned long long*>(rows);
        mp.world = world;
        mp.my = my;
        mp.n_global = s->n_global;
        mp.k = k;
        mp.min_len = min_len;
        mp.mcov = p->mcov_out;
        mp.pval = p->pval;
        mp.own_global_off = s->global_off;
        mp.out = s->d_mout;
        mp.pf_list = s->d_pf_list;
        mp.pf_cap = s->pf_cap;
        mp.res = s->d_res;
        const char* where = "k_merge_stats";
        cudaError_t e = launch_merge_stats(mp, c->stream);
        c->timer.end(c->stream);
        c->launches += 2;
        // phase 2 from the survivor list, its length and max_clust_length read on the device
        e2s_snp_counts counts;
        if (e == cudaSuccess) {
            where = "phase 2 kernels";
            e = snp_run(s->work, a, *p, E2S_MAX_C_LEN, c->d_bases, c->d_off, c->n_reads, c->sm_count, c->stream, &counts, &c->launches, &err,
                        &c->timer, s->d_pf_list, s->pf_cap, &s->d_res->n_pf, &s->d_mout->total.max_clust_length, false);
        }
        if (e == cudaSuccess) {
            where = "copy of the scan accumulators";
            e = cudaMemcpyAsync(&h, s->d_res, sizeof h, cudaMemcpyDeviceToHost, c->stream);
        }
        if (e == cudaSuccess) {
            where = "copy of the merge result";
            e = cudaMemcpyAsync(&mo, s->d_mout, sizeof mo, cudaMemcpyDeviceToHost, c->stream);
        }
        if (e == cudaSuccess && cm) {
            where = "copy of the exchange rows";
            e = cudaMemcpyAsync(cm->h_recv, cm->d_recv, size_t(world) * XR_WORDS * 8, cudaMemcpyDeviceToHost, c->stream);
        }
        if (e == cudaSuccess) {
            where = "synchronisation of the step";
            e = cudaStreamSynchronize(c->stream);  // the only synchronisation of the step
        }
        if (e != cudaSuccess) {
            rc = cuda_fail(c, e, err && err[0] ? err : where);
            break;
        }
        // a full record segment (on any rank: every rank sees every row) or a full survivor list: more room, once more
        bool any_overflow = h.overflow != 0;
        if (cm)
            for (int g = 0; g < world; ++g) any_overflow |= reinterpret_cast<const ClusterDev*>(cm->h_recv + size_t(g) * XR_WORDS)->overflow != 0;
        const bool pf_overflow = h.n_pf > s->pf_cap || (h.overflow & 2);
        if (any_overflow || pf_overflow) {
            if (attempt >= 2) {
                rc = fail(c, E2S_ERR_STATE, "record / survivor buffers still too small after two resizes");
                break;
            }
            if ((h.overflow & 1) && (rc = s->last_one_pass ? grow_segments(s) : ensure_records(s, h.n_written + 4096))) break;
            if (pf_overflow) s->pf_want = h.n_pf + h.n_pf / 8 + 4096;
            continue;
        }
        if (mo.status != MERGE_OK) {
            rc = fail(c, merge_status(mo.status), mo.status == MERGE_EMPTY ? "no clusters (the reference divides by zero here)" : merge_message(mo.status));
            break;
        }
        cudaError_t src = cudaSuccess;
        if (!snp_collect(s->work, &counts, &err, &src)) {
            if (src == cudaSuccess)  // a capacity guess of phase 2 was too small: the lists it starts from are still on the device
                src = snp_run(s->work, a, *p, mo.total.max_clust_length, c->d_bases, c->d_off, c->n_reads, c->sm_count, c->stream, &counts,
                              &c->launches, &err, &c->timer, s->d_pf_list, s->pf_cap, &s->d_res->n_pf, nullptr, true);
            if (src == cudaErrorInvalidValue && err && strstr(err, "outside the staged reads")) {
                rc = fail(c, E2S_ERR_UNSUPPORTED, err);
                break;
            }
            if (src != cudaSuccess) {
                rc = cuda_fail(c, src, err);
                break;
            }
        }
        counts.n_analysed = analysed_count(h, mo.mine, p->mcov_out, mo.total.max_clust_length);
        *cnt_out = counts;
        break;
    }
    s->pf_arm = arm_before;
    if (rc) return rc;
    // the shard's state, as e2s_cluster_run + e2s_cluster_finalize + e2s_find_events leave it
    s->h_res = h;
    s->pf_mcov = uint32_t(p->mcov_out);
    s->pf_count = h.n_pf;
    s->pf_ok = true;
    s->pf_has_adopted = true;
    s->have_scan_stats = true;
    s->m_own = h.n_written;
    s->merged = mo.mine;
    s->m_list = s->m_own + mo.mine.n_adopt;
    s->contiguous = !s->last_one_pass;
    s->adopt_put = false;
    s->have_clusters = true;
    s->staged = false;
    s->finalized = true;
    s->n_variants = cnt_out->n_variants;
    s->events_expanded = false;
    s->have_events = true;
    *mg_out = mo.mine;
    *st_out = mo.total;
    return E2S_OK;
}

// phase 2 of a pipeline on the shard's finalized records: e2s_find_events, the candidates' bytes and (events != NULL) the events
// to the caller
static int events_to_caller(e2s_shard* s, const e2s_snp_params* p, int max_clust_length, e2s_event* events, uint64_t cap_events,
                            e2s_pipeline_result* res) {
    int rc;
    res->max_clust_length = max_clust_length;
    if ((rc = e2s_find_events(s, p, max_clust_length, &res->snp))) return rc;
    res->d2h_bytes += res->snp.n_candidates * snp_event_stride(s->work);
    if (events) {
        uint64_t nv = 0;
        if ((rc = e2s_events_fetch(s, events, cap_events, &nv))) return rc;
    }
    return E2S_OK;
}

// the same after statistics() of the shard's records (res->n_written already set: an empty .clusters is refused)
static int phase2_to_caller(e2s_shard* s, const e2s_snp_params* p, e2s_event* events, uint64_t cap_events, e2s_pipeline_result* res) {
    if (res->n_written == 0) return fail(s->ctx, E2S_ERR_UNSUPPORTED, "no clusters (the reference divides by zero here)");
    e2s_stats st;
    int rc;
    if ((rc = e2s_statistics(s, &st))) return rc;
    if ((rc = e2s_statistics_finish(&st, st.last_len, p->mcov_out, p->pval))) {
        s->ctx->err = g_err;
        return rc;
    }
    return events_to_caller(s, p, st.max_clust_length, events, cap_events, res);
}

// ebwt2clust + clust2snp on a sealed shard that holds the whole eBWT of one GPU, reads already staged
int e2s_pipeline_resident(e2s_shard* s, uint32_t k, int32_t min_len, const e2s_snp_params* p, e2s_pipeline_result* res) {
    if (!s || !p || !res) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    int rc;
    const uint64_t h2d = res->h2d_bytes, d2h = res->d2h_bytes;
    memset(res, 0, sizeof *res);
    res->h2d_bytes = h2d;
    res->d2h_bytes = d2h;
    if (s->global_off != 0 || s->n_local != s->n_global)
        return fail(c, E2S_ERR_ARG, "e2s_pipeline_resident needs the whole eBWT in one shard; use e2s_pipeline_sharded");
    // both phases in one call: the scan runs clust2snp's BWT prefilter while it writes the records and the step never leaves
    // the stream (pipeline_step).  E2S_NO_FUSED_PREFILTER keeps the two phases apart as the CLIs have to.
    if (!(getenv("E2S_NO_FUSED_PREFILTER") || p->mcov_out < 1 || 2 * p->mcov_out > E2S_MAX_C_LEN)) {
        e2s_cluster_merged mg;
        e2s_stats st;
        if ((rc = pipeline_step(s, nullptr, k, min_len, p, &mg, &st, &res->snp))) return rc;
        res->n_written = mg.total_written;
        res->n_clust_out = mg.n_clust_out;
        res->max_clust_length = st.max_clust_length;
        res->d2h_bytes += res->snp.n_candidates * snp_event_stride(s->work);
        return E2S_OK;
    }
    rc = e2s_cluster_lm(s, k, min_len, &res->n_written, &res->n_clust_out);
    if (rc) return rc;
    return phase2_to_caller(s, p, nullptr, 0, res);
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

// Host-only: what every rank does with the all-gathered exchange rows (one per shard: the scan's device accumulators
// + the shard's range) -- turn them into summaries and own-record statistics, then e2s_exchange_finish.
uint64_t e2s_exchange_row_words(void) { return XR_WORDS; }

int e2s_exchange_rows_finish(const uint64_t* rows, int n_shards, int my, uint64_t n_global, uint32_t k, int32_t min_len, int mcov_out,
                             double pval, e2s_cluster_merged* mine, e2s_stats* total) {
    if (!rows || !mine || !total || n_shards < 1 || my < 0 || my >= n_shards)
        return fail(nullptr, E2S_ERR_ARG, "e2s_exchange_rows_finish: bad argument");
    const size_t ns = static_cast<size_t>(n_shards);
    std::vector<e2s_cluster_summary> sums(ns);
    std::vector<e2s_stats> own(ns);
    for (int g = 0; g < n_shards; ++g) {
        const uint64_t* row = rows + size_t(g) * XR_WORDS;
        ClusterDev h;
        memcpy(&h, row, sizeof h);
        make_summary(h, row[XR_DEV_WORDS + 0], row[XR_DEV_WORDS + 1], n_global, k, min_len, row[XR_DEV_WORDS + 2], &sums[size_t(g)]);
        e2s_stats& o = own[size_t(g)];
        memset(&o, 0, sizeof o);
        for (int i = 0; i < E2S_HIST_BINS; ++i) o.hist[i] = h.hist[i];
        o.n_bases = h.n_bases;
        o.n_clust = h.n_written;
        o.last_len = h.last_rec & 0xffff;
    }
    return e2s_exchange_finish(sums.data(), own.data(), n_shards, my, mcov_out, pval, mine, total);
}

// The sharded step in one call: K1, K2, ONE all-gather of the scan accumulators (summary + own length histogram) on
// the stream, host merge of all shards + statistics, K3/K4 on local data.  Two host synchronisations, like the
// single-shard e2s_pipeline_resident.
int e2s_pipeline_sharded(e2s_shard* s, e2s_comm* cm, uint32_t k, int32_t min_len, const e2s_snp_params* p, e2s_cluster_merged* mg,
                         e2s_stats* st, e2s_snp_counts* cnt) {
    if (!s || !cm || !p || !mg || !st || !cnt) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_pipeline_sharded: NULL argument");
    e2s_ctx* c = s->ctx;
    if (cm->ctx != c) return fail(c, E2S_ERR_ARG, "e2s_pipeline_sharded: communicator belongs to another context");
    // the exchange between the phases stays on the device: ncclAllGather of the rows, k_merge_stats on every rank (pipeline_step)
    if (!(getenv("E2S_NO_FUSED_PREFILTER") || p->mcov_out < 1 || 2 * p->mcov_out > E2S_MAX_C_LEN)) return pipeline_step(s, cm, k, min_len, p, mg, st, cnt);
    e2s_cluster_summary own_sum;
    int rc = cluster_run_impl(s, k, min_len, &own_sum, cm);
    if (rc) return rc;
    if ((rc = e2s_exchange_rows_finish(cm->h_recv, cm->world, cm->rank, s->n_global, k, min_len, p->mcov_out, p->pval, mg, st))) {
        c->err = g_err;
        return rc;
    }
    if ((rc = e2s_cluster_finalize(s, mg))) return rc;
    return e2s_find_events(s, p, st->max_clust_length, cnt);
}

// forget the chunks scanned so far: the shard is about to stream its range again (or another data set of the same shape)
int e2s_chunked_reset(e2s_shard* s) {
    if (!s || !s->chunked) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunked_reset: not a chunked shard");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    memset(&s->acc, 0, sizeof s->acc);
    s->carry_state = s->range_lo == 0 ? 0 : 1;
    s->pay_used = s->surv_count = 0;
    s->chunk_open = s->records_flushed = false;
    s->have_clusters = s->have_events = s->finalized = false;
    s->pf_ok = false;
    s->global_off = s->range_lo;
    s->n_local = s->chunk_cap < s->range_n ? s->chunk_cap : s->range_n;
    CU(c, cudaMemsetAsync(s->d_cap_counters, 0, 4 * 8, c->stream));
    return E2S_OK;
}

static uint64_t chunk_positions_from_env() {
    uint64_t chunk = uint64_t(1) << 28;  // 3.5 GB of 13-byte records per chunk, 3.9 GB of device buffers
    if (const char* e = getenv("E2S_CHUNK_POSITIONS")) {
        const uint64_t v = strtoull(e, nullptr, 10);
        if (v) chunk = v;
    }
    return chunk;
}

// the reads of a pipeline call (bases == NULL: those staged before), queued first on the stream; the scan kernels do not wait
// for them
static int stage_reads(e2s_ctx* c, const uint8_t* bases, const uint64_t* off, uint64_t n_reads, e2s_pipeline_result* res) {
    if (!bases) return E2S_OK;
    if (int rc = e2s_reads_stage(c, bases, off, n_reads)) return rc;
    res->h2d_bytes += off[n_reads] + (n_reads + 1) * 8;
    return E2S_OK;
}

// the context's cached chunked shard for the range [range_lo, range_lo + range_n) of an eBWT of n_global positions, in chunks of
// E2S_CHUNK_POSITIONS: reset for another pass when it has that shape, else made anew
static int cached_chunked(e2s_ctx* c, uint64_t range_lo, uint64_t range_n, uint64_t n_global, e2s_shard** out) {
    const uint64_t chunk = chunk_positions_from_env();
    e2s_shard* s = c->cached;
    int rc;
    if (!s || !s->chunked || s->range_lo != range_lo || s->range_n != range_n || s->n_global != n_global ||
        s->chunk_cap != chunk_buffer_positions(chunk, range_n)) {
        if (s) e2s_shard_destroy(s);
        c->cached = nullptr;
        if ((rc = e2s_shard_create_chunked(c, range_n, range_lo, n_global, chunk, &s))) return rc;
        c->cached = s;
    } else if ((rc = e2s_chunked_reset(s))) {
        return rc;
    }
    *out = s;
    return E2S_OK;
}

// chunk `lo` of a chunked shard's range: returns its length; [*a, *b) = the global positions its loads cover -- PAD_L of left
// context (from `first`, the first position the caller holds, on) to the right halo, inside the eBWT
static uint64_t chunk_window(const e2s_shard* s, uint64_t lo, uint64_t first, uint64_t* a, uint64_t* b) {
    const uint64_t end = s->range_lo + s->range_n;
    const uint64_t cn = end - lo < s->chunk_cap ? end - lo : s->chunk_cap;
    const uint64_t a0 = lo >= uint64_t(PAD_L) ? lo - PAD_L : 0;
    *a = a0 > first ? a0 : first;
    *b = lo + cn + MAX_C_LEN + 1 < s->n_global ? lo + cn + MAX_C_LEN + 1 : s->n_global;
    return cn;
}

// after a chunk's loads: its scan, then its records into rec10 from slot *off_rec on
static int scan_chunk_out(e2s_shard* s, uint32_t k, int32_t min_len, int mcov_out, void* rec10, uint64_t cap_records, uint64_t* off_rec,
                          e2s_pipeline_result* res) {
    int rc;
    uint64_t m = 0;
    if ((rc = e2s_chunk_scan(s, k, min_len, mcov_out, &m))) return rc;
    if (rec10) {
        if (*off_rec + m > cap_records) return fail(s->ctx, E2S_ERR_ARG, "record capacity too small");
        uint64_t got = 0;
        if (m && (rc = e2s_cluster_fetch_packed(s, static_cast<uint8_t*>(rec10) + *off_rec * 10, cap_records - *off_rec, &got))) return rc;
        res->d2h_bytes += m * 10;
    }
    *off_rec += m;
    return E2S_OK;
}

// After the last chunk of a range that is the whole eBWT: e2s_chunked_finish, e2s_cluster_merge, e2s_cluster_finalize, the records
// of the tail rule into rec10 from slot off_rec on (they come last, ref:ebwt2clust.cpp:127-135) and the counts of .clusters into
// res.  A failed step's code comes back as it is: the caller decides what E2S_ERR_UNSUPPORTED from the chunked steps means (the
// merge never returns it).
static int finish_range(e2s_shard* s, const char* who, uint32_t k, int32_t min_len, void* rec10, uint64_t cap_records, uint64_t off_rec,
                       e2s_pipeline_result* res) {
    e2s_ctx* c = s->ctx;
    int rc;
    e2s_cluster_summary sum;
    if ((rc = e2s_chunked_finish(s, k, min_len, &sum))) return rc;
    e2s_cluster_merged mg;
    if ((rc = e2s_cluster_merge(&sum, 1, 0, &mg))) {
        c->err = g_err;
        return rc;
    }
    if ((rc = e2s_cluster_finalize(s, &mg))) return rc;
    if (rec10) {
        if (off_rec + mg.n_append > cap_records) return fail(c, E2S_ERR_ARG, std::string(who) + ": record capacity too small");
        for (uint32_t i = 0; i < mg.n_append; ++i)
            put_rec10(static_cast<uint8_t*>(rec10) + (off_rec + i) * 10, mg.append_start[i], mg.append_len[i]);
    }
    res->n_written = mg.total_written;
    res->n_clust_out = mg.n_clust_out;
    return E2S_OK;
}

// the same from a resident shard (inputs the one-pass scan does not take: an LCP value above 127, -m > 33)
static int pipeline_host_resident(e2s_ctx* c, const void* gesa, uint64_t n, int x, int y, int z, uint32_t k, int32_t min_len,
                                  const e2s_snp_params* p, void* rec10, uint64_t cap_records, e2s_event* events, uint64_t cap_events,
                                  e2s_pipeline_result* res) {
    int rc;
    e2s_shard* s = c->cached;
    if (!s || s->chunked || s->n_local != n || s->n_global != n) {
        if (s) e2s_shard_destroy(s);
        c->cached = nullptr;
        rc = e2s_shard_create(c, n, 0, n, &s);
        if (rc) return rc;
        c->cached = s;
    }
    const int rs = x + y + z + 1;
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));  // a cached shard is reloaded from its first position: forget the old verdict
    if ((rc = e2s_shard_load_gesa(s, gesa, 0, n, x, y, z))) return rc;
    if ((rc = e2s_shard_seal(s))) return rc;
    res->h2d_bytes += n * uint64_t(rs);
    if ((rc = e2s_pipeline_resident(s, k, min_len, p, res))) return rc;
    if (rec10) {
        uint64_t m = 0;
        if ((rc = e2s_cluster_fetch_packed(s, rec10, cap_records, &m))) return rc;
        res->d2h_bytes += m * 10;
    }
    if (events) {
        uint64_t nv = 0;
        if ((rc = e2s_events_fetch(s, events, cap_events, &nv))) return rc;
    }
    return E2S_OK;
}

// All chunks of a chunked shard's range from host records (`records` = the record of global position `first`; it must reach
// from the range's left context to its right halo): load, scan, this chunk's records out (into rec10 from slot *off_rec on).
static int stream_range(e2s_shard* s, const void* records, uint64_t first, int x, int y, int z, uint32_t k, int32_t min_len,
                        int mcov_out, void* rec10, uint64_t cap_records, uint64_t* off_rec, e2s_pipeline_result* res) {
    const uint64_t end = s->range_lo + s->range_n;
    const int rs = x + y + z + 1;
    const uint8_t* src = static_cast<const uint8_t*>(records);
    int rc;
    for (uint64_t lo = s->range_lo; lo < end; lo += s->chunk_cap) {
        uint64_t a, b;
        const uint64_t cn = chunk_window(s, lo, first, &a, &b);
        if ((rc = e2s_chunk_begin(s, lo, cn))) return rc;
        if ((rc = e2s_shard_load_gesa(s, src + (a - first) * uint64_t(rs), a, b - a, x, y, z))) return rc;
        res->h2d_bytes += (b - a) * uint64_t(rs);
        if ((rc = scan_chunk_out(s, k, min_len, mcov_out, rec10, cap_records, off_rec, res))) return rc;
    }
    return E2S_OK;
}

// ebwt2clust + clust2snp from host buffers.  The records stream through a CHUNKED shard (a chunk is a shard in time): the
// device holds one chunk of E2S_CHUNK_POSITIONS positions (default 2^28) whatever n is, the H2D copies of a chunk run on
// their own stream ahead of its de-interleave kernels, each chunk's records go back as soon as it is scanned, the records
// of the clusters that survive the fused prefilter are kept for phase 2, which runs once after the last chunk.
int e2s_pipeline_host(e2s_ctx* c, const void* gesa, uint64_t n, int x, int y, int z, const uint8_t* read_bases,
                      const uint64_t* read_off, uint64_t n_reads, uint32_t k, int32_t min_len, const e2s_snp_params* p,
                      void* rec10, uint64_t cap_records, e2s_event* events, uint64_t cap_events, e2s_pipeline_result* res) {
    if (!c || !gesa || !p || !res) return fail(c, E2S_ERR_ARG, "NULL argument");
    memset(res, 0, sizeof *res);
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    if (n < 2) return fail(c, E2S_ERR_ARG, "e2s_pipeline_host: need at least 2 records");
    if ((rc = stage_reads(c, read_bases, read_off, n_reads, res))) return rc;
    const bool mcov_ok = p->mcov_out >= 1 && 2 * p->mcov_out <= E2S_MAX_C_LEN;
    if (min_len > 33 || !mcov_ok || getenv("E2S_NO_FUSED_PREFILTER"))
        return pipeline_host_resident(c, gesa, n, x, y, z, k, min_len, p, rec10, cap_records, events, cap_events, res);
    e2s_shard* s;
    if ((rc = cached_chunked(c, 0, n, n, &s))) return rc;
    // An input the streamed path refuses, whichever chunk finds it -- an LCP value above 127 under -k > 127, a cluster of
    // 65 536 positions or more whose wrapped length passes the filters and whose start has left the device -- goes through
    // a resident shard from the first record on: the records and counts of the streamed attempt are dropped.
    const uint64_t reads_h2d = res->h2d_bytes;
    auto resident = [&]() {
        memset(res, 0, sizeof *res);
        res->h2d_bytes = reads_h2d;
        return pipeline_host_resident(c, gesa, n, x, y, z, k, min_len, p, rec10, cap_records, events, cap_events, res);
    };
    uint64_t off_rec = 0;
    rc = stream_range(s, gesa, 0, x, y, z, k, min_len, p->mcov_out, rec10, cap_records, &off_rec, res);
    if (rc == E2S_OK) rc = finish_range(s, "e2s_pipeline_host", k, min_len, rec10, cap_records, off_rec, res);
    if (rc == E2S_ERR_UNSUPPORTED) return resident();
    if (rc) return rc;
    // (outside the fall-back: "no clusters" is E2S_ERR_UNSUPPORTED too, and returned as it is)
    return phase2_to_caller(s, p, events, cap_events, res);
}


// ebwt2clust + clust2snp from the BCR triple in host memory, lean: only X.out.lcp (x bytes per position) and X.out (1 byte) are
// copied to the device in full; X.out.pairSA stays on the host and only the survivors' records are fetched from it.  Same
// outputs as e2s_pipeline_host on the same index.  Needs the one-pass scan (-m <= 33; -k <= 127 when an LCP value exceeds 127) and 2 <= 2 mcov <= 150.
int e2s_pipeline_host_soa(e2s_ctx* c, const void* lcp, int x, const uint8_t* bwt, const void* pair_sa, int y, int z, uint64_t n,
                          const uint8_t* read_bases, const uint64_t* read_off, uint64_t n_reads, uint32_t k, int32_t min_len,
                          const e2s_snp_params* p, void* rec10, uint64_t cap_records, e2s_event* events, uint64_t cap_events,
                          e2s_pipeline_result* res) {
    if (!c || !lcp || !bwt || !pair_sa || !p || !res) return fail(c, E2S_ERR_ARG, "NULL argument");
    memset(res, 0, sizeof *res);
    if (n < 2) return fail(c, E2S_ERR_ARG, "e2s_pipeline_host_soa: need at least 2 records");
    const bool mcov_ok = p->mcov_out >= 1 && 2 * p->mcov_out <= E2S_MAX_C_LEN;
    if (min_len > 33 || !mcov_ok) return fail(c, E2S_ERR_UNSUPPORTED, "e2s_pipeline_host_soa: needs -m <= 33 and 1 <= mcov_out <= 75");
    int rc;
    if ((rc = stage_reads(c, read_bases, read_off, n_reads, res))) return rc;
    e2s_shard* s;
    if ((rc = cached_chunked(c, 0, n, n, &s))) return rc;
    if ((rc = e2s_shard_host_gsa(s, pair_sa, y, z))) return rc;
    if ((rc = e2s_shard_set_layout(s, x, y, z, 1))) return rc;
    s->lean_h2d = s->lean_d2h = 0;
    uint64_t off_rec = 0;
    const uint8_t* lsrc = static_cast<const uint8_t*>(lcp);
    // The lcp + BWT bytes of chunk i + 1 cross PCIe on the copy stream, into one of two staging buffers, while chunk i is widened
    // (from its staging buffer), scanned, its records fetched and its survivors' records gathered from the host's pairSA.
    const uint64_t span = s->chunk_cap + PAD_L + MAX_C_LEN + 1;  // positions a chunk loads at most
    const size_t stage_bytes = size_t(span) * size_t(x + 1) + 256;
    if (c->soa_stage_cap < stage_bytes) {
        CU(c, cudaStreamSynchronize(c->stream));
        for (int i = 0; i < 2; ++i) {
            cudaFree(c->d_soa_stage[i]);
            c->d_soa_stage[i] = nullptr;
        }
        c->soa_stage_cap = 0;
        for (int i = 0; i < 2; ++i)
            if (cudaMalloc(reinterpret_cast<void**>(&c->d_soa_stage[i]), stage_bytes) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "SoA staging buffers");
        c->soa_stage_cap = stage_bytes;
    }
    if ((rc = ensure_copy_stream(c))) return rc;
    for (int i = 0; i < 2; ++i) {
        if (!c->ev_soa_staged[i]) CU(c, cudaEventCreateWithFlags(&c->ev_soa_staged[i], cudaEventDisableTiming));
        if (!c->ev_soa_free[i]) CU(c, cudaEventCreateWithFlags(&c->ev_soa_free[i], cudaEventDisableTiming));
    }
    auto stage = [&](uint64_t lo, int buf, bool reused) -> cudaError_t {  // lcp bytes, then (64-byte aligned) the BWT bytes
        uint64_t a, b;
        chunk_window(s, lo, 0, &a, &b);
        cudaError_t e = cudaSuccess;
        if (reused) e = cudaStreamWaitEvent(c->copy_stream, c->ev_soa_free[buf], 0);
        uint8_t* d = c->d_soa_stage[buf];
        if (e == cudaSuccess) e = cudaMemcpyAsync(d, lsrc + a * uint64_t(x), (b - a) * uint64_t(x), cudaMemcpyHostToDevice, c->copy_stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d + round_up((b - a) * uint64_t(x), 64), bwt + a, b - a, cudaMemcpyHostToDevice, c->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(c->ev_soa_staged[buf], c->copy_stream);
        return e;
    };
    CU(c, stage(0, 0, false));
    uint64_t ci = 0;
    for (uint64_t lo = 0; lo < n; lo += s->chunk_cap, ++ci) {
        uint64_t a, b;
        const uint64_t cn = chunk_window(s, lo, 0, &a, &b);
        const int buf = int(ci & 1);
        if (lo + s->chunk_cap < n) {
            const cudaError_t e = stage(lo + s->chunk_cap, buf ^ 1, ci >= 1);
            if (e != cudaSuccess) {
                rc = cuda_fail(c, e, "e2s_pipeline_host_soa: staging");
                break;
            }
        }
        if ((rc = e2s_chunk_begin(s, lo, cn))) break;
        CU(c, cudaStreamWaitEvent(c->stream, c->ev_soa_staged[buf], 0));
        const uint8_t* d = c->d_soa_stage[buf];
        if ((rc = load_lcp_bwt(s, d, x, d + round_up((b - a) * uint64_t(x), 64), a, b - a, true))) break;
        CU(c, cudaEventRecord(c->ev_soa_free[buf], c->stream));
        if ((rc = e2s_shard_set_layout(s, x, y, z, 1))) break;
        res->h2d_bytes += (b - a) * uint64_t(x + 1);
        if ((rc = scan_chunk_out(s, k, min_len, p->mcov_out, rec10, cap_records, &off_rec, res))) break;
    }
    if (rc) cudaStreamSynchronize(c->copy_stream);  // (a staged copy may still be reading the caller's buffers)
    e2s_shard_host_gsa(s, nullptr, 4, 4);  // (the caller's buffer is not ours to keep)
    if (rc) return rc;
    res->h2d_bytes += s->lean_h2d;
    res->d2h_bytes += s->lean_d2h;
    if ((rc = finish_range(s, "e2s_pipeline_host_soa", k, min_len, rec10, cap_records, off_rec, res))) return rc;
    return phase2_to_caller(s, p, events, cap_events, res);
}

// After the last chunk of every rank's chunked shard: e2s_chunked_finish, ONE ncclAllGather of the ranks' rows (accumulators +
// range, the format of the resident sharded step), merge + statistics() on every rank, e2s_cluster_finalize.  Collective.
int e2s_chunked_exchange(e2s_shard* s, e2s_comm* cm, uint32_t k, int32_t min_len, int mcov_out, double pval, e2s_cluster_merged* merged,
                         e2s_stats* stats) {
    if (!s || !cm || !merged || !stats) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunked_exchange: NULL argument");
    e2s_ctx* c = s->ctx;
    if (cm->ctx != c) return fail(c, E2S_ERR_ARG, "e2s_chunked_exchange: communicator belongs to another context");
    int rc;
    e2s_cluster_summary sum;
    if ((rc = e2s_chunked_finish(s, k, min_len, &sum))) return rc;
    uint64_t row[XR_WORDS];
    memcpy(row, &s->acc, sizeof(ClusterDev));
    reinterpret_cast<ClusterDev*>(row)->ticket = 0;
    row[XR_DEV_WORDS + 0] = s->range_n;
    row[XR_DEV_WORDS + 1] = s->range_lo;
    row[XR_DEV_WORDS + 2] = uint64_t(s->lay_x);
    row[XR_DEV_WORDS + 3] = 0;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemcpyAsync(cm->d_send, row, sizeof row, cudaMemcpyHostToDevice, c->stream));
    if ((rc = all_gather_rows(c, cm))) return rc;
    CU(c, cudaMemcpyAsync(cm->h_recv, cm->d_recv, size_t(cm->world) * XR_WORDS * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if ((rc = e2s_exchange_rows_finish(cm->h_recv, cm->world, cm->rank, s->n_global, k, min_len, mcov_out, pval, merged, stats))) {
        c->err = g_err;
        return rc;
    }
    return e2s_cluster_finalize(s, merged);
}

// One eBWT over the GPUs of a box, from host buffers, one process (rank) per GPU: every rank streams ITS range of the records
// through a chunked shard (staging nothing but its range + halo), the ranks' summaries and own-record histograms are
// all-gathered (one ncclAllGather of a row per rank), every rank merges and finishes statistics(), then runs phase 2 on its
// captured survivors.  `records` = the record of global position `first`; the buffer must reach from max(0, range_lo - 176)
// to min(n_global, range_lo + range_n + 152).  rec10 receives this rank's slice of .clusters (head record, own records,
// tail records, in file order): *n_records records that belong at index merged->record_offset of the file.
int e2s_pipeline_host_sharded(e2s_ctx* c, e2s_comm* cm, const void* records, uint64_t first, uint64_t range_lo, uint64_t range_n,
                              uint64_t n_global, int x, int y, int z, const uint8_t* read_bases, const uint64_t* read_off,
                              uint64_t n_reads, uint32_t k, int32_t min_len, const e2s_snp_params* p, void* rec10,
                              uint64_t cap_records, uint64_t* n_records, e2s_event* events, uint64_t cap_events,
                              e2s_cluster_merged* merged, e2s_stats* stats, e2s_pipeline_result* res) {
    if (!c || !cm || !records || !p || !res || !merged || !stats) return fail(c, E2S_ERR_ARG, "NULL argument");
    if (cm->ctx != c) return fail(c, E2S_ERR_ARG, "e2s_pipeline_host_sharded: communicator belongs to another context");
    memset(res, 0, sizeof *res);
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    if (!(p->mcov_out >= 1 && 2 * p->mcov_out <= E2S_MAX_C_LEN) || min_len > 33)
        return fail(c, E2S_ERR_UNSUPPORTED, "e2s_pipeline_host_sharded needs a valid -m (clust2snp) and ebwt2clust -m <= 33");
    if ((rc = stage_reads(c, read_bases, read_off, n_reads, res))) return rc;
    e2s_shard* s;
    if ((rc = cached_chunked(c, range_lo, range_n, n_global, &s))) return rc;
    uint8_t* out = static_cast<uint8_t*>(rec10);
    uint64_t off_rec = rec10 ? 1 : 0;  // slot 0 is kept for the shard's head record
    if ((rc = stream_range(s, records, first, x, y, z, k, min_len, p->mcov_out, rec10, cap_records, &off_rec, res))) return rc;
    if ((rc = e2s_chunked_exchange(s, cm, k, min_len, p->mcov_out, p->pval, merged, stats))) return rc;
    uint64_t slice_first = 1, m_slice = off_rec ? off_rec - 1 : 0;
    if (rec10) {
        if (merged->n_prepend && merged->prepend_written) {
            put_rec10(out, merged->prepend_start, merged->prepend_len);
            slice_first = 0;
            ++m_slice;
        }
        if (off_rec + merged->n_append > cap_records) return fail(c, E2S_ERR_ARG, "record capacity too small");
        for (uint32_t i = 0; i < merged->n_append; ++i) put_rec10(out + (off_rec + i) * 10, merged->append_start[i], merged->append_len[i]);
        m_slice += merged->n_append;
        if (slice_first) memmove(out, out + 10, size_t(m_slice) * 10);  // no head record: the slice starts at slot 0 all the same
    }
    if (n_records) *n_records = m_slice;
    res->n_written = merged->total_written;
    res->n_clust_out = merged->n_clust_out;
    return events_to_caller(s, p, stats->max_clust_length, events, cap_events, res);
}

}  // extern "C"
