// Host side of the C ABI (include/ebwt2snp_b200.h): contexts, shards and communicators, the error convention, and the
// helpers more than one of its translation units calls (ctx.cu, shard.cu, build_host.cu, phase1.cu, phase2.cu, pipeline.cu).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <functional>
#include <initializer_list>
#include <string>
#include <vector>

#include "common.cuh"
#include "internal.h"

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
    e2s::KernelTimer timer;
};

namespace e2s {

constexpr uint64_t GSA_TAIL = 512;  // lean SoA mode: text / suff of the last positions of the eBWT are loaded like the rest (phantom records, tail clusters)

// What a shard's record list currently is.  The fields are read directly and written only by the functions below, one per
// outcome of a call; each leaves the fields it does not name as they were.
struct RecordList {
    uint64_t m_own = 0;     // records produced by the scan (or staged)
    uint64_t m_list = 0;    // records phase 2 analyses = own + adopted
    bool have_clusters = false, staged = false, finalized = false;
    e2s_cluster_merged merged;
    bool contiguous = true;          // d_start / d_len hold the record list (false: it still lies in the segments)
    bool adopt_put = false;          // the records adopted from the merge have been appended to d_start / d_len
    bool records_flushed = false;    // e2s_chunked_finish ran: the records were handed out chunk by chunk
    ClusterDev h_res;                // host copy of the last scan's accumulators (incl. length histogram)
    bool have_scan_stats = false;
    bool have_events = false;
    // the fused prefilter's survivor list (e2s_shard::d_pf_list)
    uint32_t pf_mcov = 0;            // what the last scan used
    uint64_t pf_count = 0;
    bool pf_ok = false;              // the list is complete (no overflow) and belongs to the current record list
    bool pf_has_adopted = false;     // ... and already holds the records adopted from the merge (k_merge_stats appended them)

    // records scanned, with the prefilter of -m `mcov` (0: none): h = the scan's accumulators; the own records lie in d_start /
    // d_len when `contig`, else in the scan's segments.  Not merged yet.
    void scanned(const ClusterDev& h, uint32_t mcov, bool contig) {
        h_res = h;
        pf_mcov = mcov;
        m_own = m_list = h.n_written;
        contiguous = contig;
        have_clusters = true;
        staged = false;
        finalized = false;
        have_events = false;
        have_scan_stats = true;
        memset(&merged, 0, sizeof merged);
    }
    // the survivor list the scan left: n entries, complete or not, with or without the adopted records
    void survivors(uint64_t n, bool ok, bool has_adopted) {
        pf_count = n;
        pf_ok = ok;
        pf_has_adopted = has_adopted;
    }
    // the adopted records joined the survivors: n more entries in d_pf_list (0: they went to the payload of a chunked shard)
    void survivors_adopted(uint64_t n) {
        pf_count += n;
        pf_has_adopted = true;
    }
    // one chunk's clusters staged from a .clusters file and prefiltered with -m `mcov`
    void chunk_staged(uint32_t mcov) { pf_mcov = mcov; }
    // m records staged from a .clusters file, final as they are.  captured == null: the whole list, in d_start / d_len
    // (e2s_clusters_stage).  Else a chunked shard's range after its last chunk: phase 2 runs on the records its chunks
    // captured, *captured = the range's accumulators (the length histogram of the staged records: n_analysed)
    void file_staged(uint64_t m, const ClusterDev* captured) {
        m_own = m_list = m;
        have_clusters = true;
        finalized = true;
        have_events = false;
        have_scan_stats = false;
        memset(&merged, 0, sizeof merged);
        if (captured) {
            h_res = *captured;
            records_flushed = true;
            staged = false;
            pf_ok = true;
            pf_has_adopted = true;
        } else {
            contiguous = true;
            staged = true;
            pf_ok = false;
        }
    }
    // the last chunk of a chunked shard's range was scanned: acc = the accumulators of the whole range (statistics() of it)
    void range_finished(const ClusterDev& acc) {
        h_res = acc;
        m_own = m_list = acc.n_written;
        records_flushed = true;
        pf_ok = pf_mcov != 0;
        pf_has_adopted = false;
    }
    // the merge's view of this shard applied: the adopted records join the device list when a pass over it needs them
    void finalize(const e2s_cluster_merged& mg) {
        merged = mg;
        m_list = m_own + mg.n_adopt;
        adopt_put = false;
        finalized = true;
    }
    // the records of the scan's segments were exported to d_start / d_len
    void exported() { contiguous = true; }
    // the adopted records were appended to d_start / d_len
    void adopted_in_list() { adopt_put = true; }
    // e2s_events_fetch has (present) or has not the events of the current record list
    void events_present(bool present) { have_events = present; }
    // a chunked shard forgets its range's records: it is about to stream the range again
    void reset() {
        records_flushed = false;
        have_clusters = have_events = finalized = false;
        pf_ok = false;
    }
};

}  // namespace e2s

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
    // built from the reads (e2s_shard_build_egsa_range): its first and last record as text << 32 | suff at full width (the stored
    // fields may be truncated), for the halo row
    uint64_t ends[2] = {0, 0};
    bool ends_known = false;
    // record list
    uint64_t* d_start = nullptr;
    uint16_t* d_len = nullptr;
    uint64_t rec_cap = 0;
    e2s::RecordList rl;
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
    e2s::ChunkRec* d_chunks = nullptr;    // SCAN_MAX_CHUNKS chunk summaries
    e2s::ChunkSeg* d_segs = nullptr;      // ... and where k_chunk_resolve put each segment in the position-ordered list
    bool last_one_pass = false;      // what the last scan used
    uint64_t pf_want = 0;            // survivor-list capacity asked for after an overflow
    uint64_t* d_row = nullptr;       // this shard's exchange row (XR_WORDS) when there is no communicator
    e2s::MergeOut* d_mout = nullptr;      // k_merge_stats output
    e2s::MergeOut* h_mout = nullptr;      // ... its pinned host copy
    e2s::ClusterDev* d_res = nullptr;
    e2s::ClusterDev* h_pin = nullptr; // pinned staging for the host copy of the scan's accumulators
    uint8_t* d_packed = nullptr;
    uint64_t packed_cap = 0;
    unsigned long long* d_hist = nullptr;
    // fused prefilter: clust2snp's -m for the next e2s_cluster_run (e2s_cluster_prefilter), 0 = plain scan
    uint32_t pf_arm = 0;
    e2s::SurvEntry* d_pf_list = nullptr;
    uint64_t pf_cap = 0;
    uint4* d_planes = nullptr;       // resident base-code bit planes of the BWT (planes.cuh), written by the loads
    uint32_t* d_seal_flag = nullptr; // != 0: an LCP value above 127 (set at seal)
    // chunked mode (streaming): the device buffers hold one chunk [global_off, global_off + n_local) of the shard's range at a time
    bool chunked = false;
    // lean SoA mode (e2s_shard_host_gsa): text / suff stay on the host in the BCR pairSA layout; only the records of the clusters
    // that reach phase 2 are fetched from there (capture_survivors), the last GSA_TAIL positions of the eBWT excepted
    const uint8_t* host_gsa = nullptr;
    int gsa_y = 4, gsa_z = 4;
    uint64_t lean_h2d = 0, lean_d2h = 0;                    // bytes of the survivor fetches (for the callers' accounting)
    e2s::SnpDev* d_stage_dev = nullptr;                      // e2s_chunk_stage_clusters: K3a's counters
    e2s::SurvEntry* h_surv = nullptr; size_t h_surv_cap = 0; // pinned
    uint32_t* h_gather = nullptr; size_t h_gather_cap = 0;  // pinned: text values then suff values of one capture
    uint64_t range_lo = 0, range_n = 0;   // the shard's own range of the eBWT
    uint64_t chunk_cap = 0;               // positions the buffers hold
    bool chunk_open = false;              // a chunk has been begun and not yet scanned
    e2s::ClusterDev acc;                  // the range's accumulators so far (host)
    uint64_t carry_state = 0;             // open-cluster state after the chunks so far: 0 closed, 1 unknown (an earlier shard decides), >= 2: 2 + global START
    uint32_t* p_lcp = nullptr;            // payload of the surviving clusters (see CaptureParams)
    uint32_t* p_text = nullptr;
    uint32_t* p_suff = nullptr;
    uint8_t* p_bwt = nullptr;
    uint64_t pay_cap = 0, pay_used = 0;
    e2s::SurvEntry* d_surv = nullptr;
    uint64_t surv_cap = 0, surv_count = 0;
    unsigned long long* d_cap_counters = nullptr;  // payload cursor, survivor count, error bits
    // phase 2
    e2s::SnpWork* work = nullptr;
    std::vector<e2s_event> events;
    uint64_t n_variants = 0;
    bool events_expanded = false;
};

struct e2s_comm {
    e2s_ctx* ctx = nullptr;
    void* nccl = nullptr;
    e2s_gather_fn fn = nullptr;  // instead of nccl: the caller's all-gather, on the host (e2s_comm_create_gather)
    void* user = nullptr;
    int rank = 0, world = 1;
    uint64_t* d_send = nullptr;  // XR_WORDS
    uint64_t* d_recv = nullptr;  // world * XR_WORDS
    uint64_t* h_recv = nullptr;  // pinned
    uint64_t* h_send = nullptr;  // pinned, XR_WORDS (fn only)
};

namespace e2s {

// The message of the last failure: every call that fails sets it, and the context's copy when there is a context.  One
// object for the whole library (ctx.cu): a host-only call that fails without a context leaves its message here only.
extern thread_local std::string g_err;

int fail(e2s_ctx* ctx, int code, const std::string& msg);
int cuda_fail(e2s_ctx* ctx, cudaError_t e, const char* what);
#define CU(ctx, x)                                      \
    do {                                                \
        cudaError_t _e = (x);                           \
        if (_e != cudaSuccess) return cuda_fail(ctx, _e, #x); \
    } while (0)

// ctx.cu
int all_gather_rows(e2s_ctx* c, e2s_comm* cm);

// shard.cu
int check_field_sizes(e2s_ctx* c, std::initializer_list<int> sizes);
uint64_t round_up(uint64_t v, uint64_t a);
uint64_t chunk_buffer_positions(uint64_t chunk_positions, uint64_t n_local);
int ensure_copy_stream(e2s_ctx* c);
int load_lcp_bwt(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, uint64_t first, uint64_t count, bool dev);
// the narrow resident copies (byte LCP, base-code bit planes) of the local positions [l, l + cnt) just written
cudaError_t derive_loaded(e2s_shard* s, int64_t l, uint64_t cnt, bool have_lcp, bool have_bwt);

// phase1.cu
void put_rec10(uint8_t* o, uint64_t start, uint64_t len);
int ensure_contiguous(e2s_shard* s);
SnpArrays shard_arrays(const e2s_shard* s);
uint64_t analysed_count(const ClusterDev& h, const e2s_cluster_merged& mg, int mcov_out, int max_clust_length);
// The scan of the shard, with the fused prefilter of clust2snp's -m `mcov` (0: none), run until its buffers held everything.
// Each attempt enqueues the scan, then `behind` (the caller's work that must follow it; may be empty), then the copy of the
// accumulators to *s->h_pin, and synchronises once.  A full record buffer is grown and the scan rerun; so is a full survivor
// list when retry_survivors.  cm != NULL: `behind` copied every rank's exchange row to cm->h_recv, and an overflow on any
// rank reruns the scan on all of them.  At most two resizes.
int run_scan(e2s_shard* s, uint32_t k, int32_t min_len, uint32_t mcov, bool retry_survivors, const e2s_comm* cm,
             const std::function<int()>& behind);
const char* merge_message(int rc);
int merge_status(int rc);

// phase2.cu
bool snp_params_ok(const e2s_snp_params* p);

}  // namespace e2s
