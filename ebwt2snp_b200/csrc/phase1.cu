// Phase 1 (ebwt2clust): the scan of a shard, resident or chunk by chunk, and the capture of the survivors' records;
// merge and finalize; the record list out to the caller, or staged from a .clusters file.

#include <stdlib.h>

#include "host_state.h"
#include "merge.cuh"

using namespace e2s;

namespace e2s {

// one record of a .clusters file: 8-byte start, 2-byte length
void put_rec10(uint8_t* o, uint64_t start, uint64_t len) {
    const uint16_t l16 = uint16_t(len);
    memcpy(o, &start, 8);
    memcpy(o + 8, &l16, 2);
}

static void get_rec10(const uint8_t* r, uint64_t* start, uint16_t* len) {
    memcpy(start, r, 8);
    memcpy(len, r + 8, 2);
}

// may k_cluster_scan run on this shard with these options?  (min_len <= 33: the bit-parallel length test; the saturated
// bit-sliced LCP compares exactly against k <= 127 whatever the values, against any k when nothing was saturated)
static bool one_pass_ok(const e2s_shard* s, uint32_t k, int32_t min_len) {
    return s->sealed && s->lcpt_ok && (!s->lcpt_sat || k <= 127u) && min_len <= 33;
}

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
int ensure_contiguous(e2s_shard* s) {
    if (s->rl.contiguous) return E2S_OK;
    e2s_ctx* c = s->ctx;
    int rc = ensure_records(s, s->rl.m_own + 8);
    if (rc) return rc;
    CU(c, launch_export_records(s->d_segs, s->n_chunks, s->seg_cap, s->d_seg_start, s->d_seg_len, s->d_start, s->d_len, nullptr, c->stream));
    ++c->launches;
    s->rl.exported();
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
SnpArrays shard_arrays(const e2s_shard* s) {
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
uint64_t analysed_count(const ClusterDev& h, const e2s_cluster_merged& mg, int mcov_out, int max_clust_length) {
    uint64_t na = 0;
    for (int l = 2 * mcov_out; l <= max_clust_length; ++l) na += h.hist[l];
    for (uint32_t i = 0; i < mg.n_adopt; ++i)
        na += int64_t(mg.adopt_len[i]) >= 2 * mcov_out && int64_t(mg.adopt_len[i]) <= max_clust_length;
    return na;
}

// The fused prefilter's survivor list for a scan whose records fill at most `records` slots (mcov == 0: none): what the scan
// kernels get in *list / *cap.
static int arm_survivors(e2s_shard* s, uint32_t mcov, uint64_t records, SurvEntry** list, uint64_t* cap) {
    *list = nullptr;
    *cap = 0;
    if (!mcov) return E2S_OK;
    uint64_t want = records / 16 + 4096;
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
            return fail(s->ctx, E2S_ERR_NOMEM, "prefilter survivor list");
        s->pf_cap = want;
    }
    *list = s->d_pf_list;
    *cap = s->pf_cap > 4 ? s->pf_cap - 4 : 0;  // (room for the records k_merge_stats adopts)
    return E2S_OK;
}

// K1 + K2 (k_lcp_flags + k_cluster_emit) on the 4-byte LCP, accumulators zeroed first: the records go to d_start / d_len.
static int enqueue_k1_k2(e2s_shard* s, uint32_t k, int32_t min_len, uint32_t mcov) {
    e2s_ctx* c = s->ctx;
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
    if (!s->d_start) {
        int rc = ensure_records(s, s->n_local / 8 + 4096);
        if (rc) return rc;
    }
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
    cudaError_t le = launch_flags(fp, s->alloc_r / 32, c->sm_count, c->stream);
    c->timer.end(c->stream);
    CU(c, le);
    ++c->launches;
    CU(c, cudaMemsetAsync(s->d_res, 0, sizeof(ClusterDev), c->stream));
    CU(c, cudaMemsetAsync(s->d_desc, 0, s->desc_cap * 8, c->stream));
    EmitParams p;
    p.s_words = s->d_flags;
    p.e_words = s->d_flags + s->flag_words;
    p.num_tiles = emit_num_tiles(s->n_local);
    p.global_off = s->global_off;
    p.n_global = s->n_global;
    p.min_len = min_len;
    p.out_start = s->d_start;
    p.out_len = s->d_len;
    p.cap = s->rec_cap - 4;  // room for adopted records
    p.desc = s->d_desc;
    p.planes = s->d_planes;
    p.pf_mcov = mcov;
    if (int rc = arm_survivors(s, mcov, s->rec_cap, &p.pf_list, &p.pf_cap)) return rc;
    p.res = s->d_res;
    const bool is_last = s->global_off + s->n_local == s->n_global;
    p.tail_lcp = is_last ? s->lcp + s->n_local - 2 : nullptr;
    p.tail_bwt = is_last ? s->bwt + s->n_local - 1 : nullptr;
    c->timer.begin(E2S_KERNEL_EMIT, c->stream);
    le = launch_emit(p, c->sm_count, c->stream);
    c->timer.end(c->stream);
    CU(c, le);
    ++c->launches;
    return E2S_OK;
}

// k_cluster_scan + k_chunk_resolve, one pass over the bit-sliced LCP, accumulators zeroed first: the records go to the
// per-chunk segments.  A chunked shard starts from the open-cluster state its earlier chunks left.
static int enqueue_one_pass(e2s_shard* s, uint32_t k, int32_t min_len, uint32_t mcov) {
    e2s_ctx* c = s->ctx;
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
    CU(c, cudaMemsetAsync(s->d_res, 0, sizeof(ClusterDev), c->stream));
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
    sp.pf_mcov = mcov;
    if (int rc = arm_survivors(s, mcov, s->seg_cap * s->n_chunks, &sp.pf_list, &sp.pf_cap)) return rc;
    sp.res = s->d_res;
    const bool is_last = s->global_off + s->n_local == s->n_global;
    sp.tail_lcp = is_last ? s->lcp + s->n_local - 2 : nullptr;
    sp.tail_bwt = is_last ? s->bwt + s->n_local - 1 : nullptr;
    CU(c, cudaMemsetAsync(s->d_chunks, 0, size_t(s->n_chunks) * sizeof(ChunkRec), c->stream));
    c->timer.begin(E2S_KERNEL_SCAN1, c->stream);
    cudaError_t le = launch_scan(sp, s->alloc_r, c->stream);
    c->timer.end(c->stream);
    CU(c, le);
    ++c->launches;
    ResolveParams rp;
    rp.chunks = s->d_chunks;
    rp.segs = s->d_segs;
    rp.n_chunks = s->n_chunks;
    rp.min_len = min_len;
    rp.global_off = s->global_off;
    rp.n_global = s->n_global;
    rp.init_state = s->chunked ? s->carry_state : (s->global_off == 0 ? 0 : 1);
    rp.planes = s->d_planes;
    rp.pf_mcov = mcov;
    rp.pf_list = sp.pf_list;
    rp.pf_cap = sp.pf_cap;
    rp.res = s->d_res;
    c->timer.begin(E2S_KERNEL_RESOLVE, c->stream);
    le = launch_chunk_resolve(rp, c->stream);
    c->timer.end(c->stream);
    CU(c, le);
    ++c->launches;
    return E2S_OK;
}

int run_scan(e2s_shard* s, uint32_t k, int32_t min_len, uint32_t mcov, bool retry_survivors, const e2s_comm* cm,
             const std::function<int()>& behind) {
    e2s_ctx* c = s->ctx;
    // One pass over the byte LCP (k_cluster_scan) whenever the shard has it and min_len allows the bit-parallel length test;
    // else the two-kernel path on the 4-byte LCP.  E2S_SCAN_LEGACY=1 forces the latter on a resident shard: a chunked shard
    // has the one-pass scan only.
    const bool one_pass = s->last_one_pass = one_pass_ok(s, k, min_len) && (s->chunked || !getenv("E2S_SCAN_LEGACY"));
    if (!s->h_pin) CU(c, cudaHostAlloc(reinterpret_cast<void**>(&s->h_pin), sizeof(ClusterDev), cudaHostAllocDefault));
    ClusterDev& h = *s->h_pin;
    for (int attempt = 0;; ++attempt) {
        int rc = one_pass ? enqueue_one_pass(s, k, min_len, mcov) : enqueue_k1_k2(s, k, min_len, mcov);
        if (!rc && behind) rc = behind();
        if (rc) return rc;
        CU(c, cudaMemcpyAsync(&h, s->d_res, sizeof h, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        // bit 0: a record buffer was full; bit 1 (or more entries than the list holds once k_merge_stats appended the
        // adopted records): the survivor list was
        const bool records_full = h.overflow & 1;
        const bool survivors_full = retry_survivors && ((h.overflow & 2) || h.n_pf > s->pf_cap);
        bool again = records_full || survivors_full;
        if (cm)  // every rank sees every rank's row: all of them repeat the round together
            for (int g = 0; g < cm->world; ++g)
                again |= (reinterpret_cast<const ClusterDev*>(cm->h_recv + size_t(g) * XR_WORDS)->overflow & (retry_survivors ? 3 : 1)) != 0;
        if (!again) return E2S_OK;
        if (attempt == 2) return fail(c, E2S_ERR_STATE, "record / survivor buffers still too small after two resizes");
        if (records_full && (rc = one_pass ? grow_segments(s) : ensure_records(s, h.n_written + 4096))) return rc;
        if (survivors_full) s->pf_want = h.n_pf + h.n_pf / 8 + 4096;
    }
}

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

// Host-only: chain the shards' open-cluster states, resolve head records, apply the tail rule with
// the post-EOF phantom record (ref:ebwt2clust.cpp:90-135; SURVEY.md §8(a) A3).
const char* merge_message(int rc) {
    switch (rc) {
        case MERGE_NOT_PARTITION: return "e2s_cluster_merge: shards are not a partition of [0, n_global)";
        case MERGE_NOT_COVER: return "e2s_cluster_merge: shards do not cover n_global";
        case MERGE_END_WITHOUT_START: return "e2s_cluster_merge: END without START (inconsistent summaries)";
        case MERGE_EMPTY: return "empty .clusters (the reference divides by zero here)";
        case MERGE_BAD_MCOV: return "2*mcov_out outside [0,150]";
        default: return "merge failed";
    }
}
int merge_status(int rc) {
    return rc == MERGE_END_WITHOUT_START ? E2S_ERR_STATE : ((rc == MERGE_EMPTY || rc == MERGE_BAD_MCOV) ? E2S_ERR_UNSUPPORTED : E2S_ERR_ARG);
}

// records of this shard in .clusters order: [head] + own + [tail]
static uint64_t out_count(const e2s_shard* s) {
    if (s->rl.staged) return s->rl.m_own;
    return s->rl.m_own + (s->rl.merged.n_prepend && s->rl.merged.prepend_written ? 1 : 0) + s->rl.merged.n_append;
}

}  // namespace e2s

extern "C" {

int e2s_cluster_prefilter(e2s_shard* s, int mcov_out) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (mcov_out < 0 || 2 * mcov_out > E2S_MAX_C_LEN) return fail(s->ctx, E2S_ERR_ARG, "e2s_cluster_prefilter: need 0 <= 2 * mcov_out <= 150");
    s->pf_arm = uint32_t(mcov_out);
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
    if ((rc = run_scan(s, k, min_len, uint32_t(mcov_out), true, nullptr, nullptr))) return rc;
    const ClusterDev& h = *s->h_pin;
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
    s->rl.scanned(h, uint32_t(mcov_out), !s->last_one_pass);
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
    if (s->acc.ticket && s->rl.pf_mcov != uint32_t(mcov_out)) return fail(c, E2S_ERR_ARG, "e2s_chunk_stage_clusters: one -m for all the chunks of a range");
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
    s->rl.chunk_staged(uint32_t(mcov_out));
    return E2S_OK;
}

// After the last chunk of the range went through e2s_chunk_stage_clusters: e2s_find_events runs on the captured records.
int e2s_chunked_clusters_finish(e2s_shard* s) {
    if (!s || !s->chunked) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunked_clusters_finish: not a chunked shard");
    e2s_ctx* c = s->ctx;
    if (s->chunk_open || s->global_off + s->n_local != s->range_lo + s->range_n || !s->acc.ticket)
        return fail(c, E2S_ERR_STATE, "e2s_chunked_clusters_finish: the last chunk of the range has not been staged");
    s->rl.file_staged(s->acc.n_written, &s->acc);
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
    s->rl.range_finished(h);
    return E2S_OK;
}

int e2s_cluster_run(e2s_shard* s, uint32_t k, int32_t min_len, e2s_cluster_summary* sum) {
    if (!s || !sum) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_cluster_run: NULL argument");
    e2s_ctx* c = s->ctx;
    if (s->chunked) return fail(c, E2S_ERR_STATE, "chunked shard: use e2s_chunk_begin / e2s_chunk_scan / e2s_chunked_finish");
    if (k == 0) return fail(c, E2S_ERR_ARG, "k must be >= 1 (the CLI maps 0 to the default 16)");
    CU(c, cudaSetDevice(c->device));
    // a full survivor list is not retried: find_events then runs its own prefilter (K3a)
    const uint32_t mcov = s->sealed ? s->pf_arm : 0;
    int rc = run_scan(s, k, min_len, mcov, false, nullptr, nullptr);
    if (rc) return rc;
    const ClusterDev& h = *s->h_pin;
    make_summary(h, s->n_local, s->global_off, s->n_global, k, min_len, uint64_t(s->lay_x), sum);
    s->rl.scanned(h, mcov, !s->last_one_pass);
    s->rl.survivors(h.n_pf, mcov != 0 && !(h.overflow & 2) && h.n_pf + 4 <= s->pf_cap, false);
    return E2S_OK;
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
    if (!s->rl.have_clusters || s->rl.staged) return fail(c, E2S_ERR_STATE, "e2s_cluster_finalize: run e2s_cluster_run first");
    CU(c, cudaSetDevice(c->device));
    s->rl.finalize(*mg);
    if (s->chunked && s->rl.pf_mcov && mg->n_adopt) {  // their records are still on the device (the range's last chunk): to the payload
        // only the lengths phase 2 analyses (2 mcov_out .. 150): any other adopted record is never read, and may be far longer
        // than the payload reserves per record or start in a chunk that has left the device
        SurvEntry extra[4];
        unsigned long long n = 0;
        for (uint32_t i = 0; i < mg->n_adopt && i < 4; ++i)
            if (mg->adopt_len[i] >= 2 * uint64_t(s->rl.pf_mcov) && mg->adopt_len[i] <= uint64_t(E2S_MAX_C_LEN))
                extra[n++] = SurvEntry{mg->adopt_start[i], mg->adopt_start[i] - s->global_off, uint32_t(mg->adopt_len[i]), 0u};
        if (n) {
            CU(c, cudaMemcpyAsync(s->d_pf_list, extra, n * sizeof(SurvEntry), cudaMemcpyHostToDevice, c->stream));
            CU(c, cudaMemcpyAsync(&s->d_res->n_pf, &n, 8, cudaMemcpyHostToDevice, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            int rc = capture_survivors(s, n);
            if (rc) return rc;
        }
        s->rl.survivors_adopted(0);
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

int e2s_cluster_count(const e2s_shard* s, uint64_t* m) {
    if (!s || !m) return fail(nullptr, E2S_ERR_ARG, "NULL argument");
    if (!s->rl.have_clusters) return fail(s->ctx, E2S_ERR_STATE, "no clusters yet");
    *m = out_count(s);
    return E2S_OK;
}

int e2s_cluster_fetch(e2s_shard* s, uint64_t* start, uint16_t* len, uint64_t cap, uint64_t* m) {
    if (!s || !start || !len || !m) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->rl.have_clusters) return fail(c, E2S_ERR_STATE, "no clusters yet");
    if (s->rl.records_flushed) return fail(c, E2S_ERR_STATE, "chunked shard: the records were handed out chunk by chunk");
    const uint64_t total = out_count(s);
    *m = total;
    if (cap < total) return fail(c, E2S_ERR_ARG, "e2s_cluster_fetch: capacity too small");
    CU(c, cudaSetDevice(c->device));
    uint64_t o = 0;
    if (!s->rl.staged && s->rl.merged.n_prepend && s->rl.merged.prepend_written) {
        start[o] = s->rl.merged.prepend_start;
        len[o] = uint16_t(s->rl.merged.prepend_len);
        ++o;
    }
    if (s->rl.m_own) {
        int rc = ensure_contiguous(s);
        if (rc) return rc;
        CU(c, cudaMemcpyAsync(start + o, s->d_start, s->rl.m_own * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(len + o, s->d_len, s->rl.m_own * 2, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        o += s->rl.m_own;
    }
    if (!s->rl.staged)
        for (uint32_t i = 0; i < s->rl.merged.n_append; ++i) {
            start[o] = s->rl.merged.append_start[i];
            len[o] = uint16_t(s->rl.merged.append_len[i]);
            ++o;
        }
    return E2S_OK;
}

int e2s_cluster_fetch_packed(e2s_shard* s, void* rec10, uint64_t cap, uint64_t* m) {
    if (!s || !rec10 || !m) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->rl.have_clusters) return fail(c, E2S_ERR_STATE, "no clusters yet");
    if (s->rl.records_flushed) return fail(c, E2S_ERR_STATE, "chunked shard: the records were handed out chunk by chunk");
    const uint64_t total = out_count(s);
    *m = total;
    if (cap < total) return fail(c, E2S_ERR_ARG, "e2s_cluster_fetch_packed: capacity too small");
    CU(c, cudaSetDevice(c->device));
    uint8_t* o = static_cast<uint8_t*>(rec10);
    auto put = [&](uint64_t st, uint64_t ln) {
        put_rec10(o, st, ln);
        o += 10;
    };
    if (!s->rl.staged && s->rl.merged.n_prepend && s->rl.merged.prepend_written) put(s->rl.merged.prepend_start, s->rl.merged.prepend_len);
    if (s->rl.m_own) {  // pack on the device, one D2H straight into the caller's buffer
        if (s->rl.m_own > s->packed_cap) {
            cudaFree(s->d_packed);
            s->d_packed = nullptr;
            s->packed_cap = 0;
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_packed), s->rl.m_own * 10 + 16) != cudaSuccess)
                return fail(c, E2S_ERR_NOMEM, "packed record buffer");
            s->packed_cap = s->rl.m_own;
        }
        if (s->rl.contiguous)
            CU(c, launch_pack_records(s->d_start, s->d_len, s->rl.m_own, s->d_packed, c->stream, c->sm_count));
        else  // straight from the scan's segments
            CU(c, launch_export_records(s->d_segs, s->n_chunks, s->seg_cap, s->d_seg_start, s->d_seg_len, nullptr, nullptr, s->d_packed, c->stream));
        ++c->launches;
        CU(c, cudaMemcpyAsync(o, s->d_packed, s->rl.m_own * 10, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        o += s->rl.m_own * 10;
    }
    if (!s->rl.staged)
        for (uint32_t i = 0; i < s->rl.merged.n_append; ++i) put(s->rl.merged.append_start[i], s->rl.merged.append_len[i]);
    return E2S_OK;
}

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
    s->rl.file_staged(m, nullptr);
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

// forget the chunks scanned so far: the shard is about to stream its range again (or another data set of the same shape)
int e2s_chunked_reset(e2s_shard* s) {
    if (!s || !s->chunked) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunked_reset: not a chunked shard");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    memset(&s->acc, 0, sizeof s->acc);
    s->carry_state = s->range_lo == 0 ? 0 : 1;
    s->pay_used = s->surv_count = 0;
    s->chunk_open = false;
    s->rl.reset();
    s->global_off = s->range_lo;
    s->n_local = s->chunk_cap < s->range_n ? s->chunk_cap : s->range_n;
    CU(c, cudaMemsetAsync(s->d_cap_counters, 0, 4 * 8, c->stream));
    return E2S_OK;
}

}  // extern "C"
