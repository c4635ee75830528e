// End to end: both phases in one call, on a resident shard (one step on the stream) or streamed from host buffers
// through a chunked shard, on one GPU or one rank per GPU.

#include <stdlib.h>

#include "host_state.h"
#include "merge.cuh"

using namespace e2s;

namespace e2s {

// may both phases run in one pass, the scan running clust2snp's BWT prefilter?  Needs a valid -m; E2S_NO_FUSED_PREFILTER
// keeps the two phases apart as the CLIs have to (e2s_pipeline_sharded always runs them in one pass).
static bool fused_prefilter(const e2s_snp_params* p) {
    return !(getenv("E2S_NO_FUSED_PREFILTER") || p->mcov_out < 1 || 2 * p->mcov_out > E2S_MAX_C_LEN);
}

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
    MergeOut& mo = *s->h_mout;
    s->rl.events_present(false);
    s->events.clear();
    const SnpArrays a = shard_arrays(s);  // (phase 2 starts from the survivor list: the record list is not walked)
    const char* err = "";
    e2s_snp_counts counts;
    // behind the scan on the stream: the exchange row (all-gathered when there is a communicator), k_merge_stats, phase 2 from the
    // survivor list -- its length and max_clust_length read on the device -- and the copies of the results
    auto merge_and_phase2 = [&]() -> int {
        uint64_t* send = cm ? cm->d_send : s->d_row;
        c->timer.begin(E2S_KERNEL_MERGE, c->stream);
        if (launch_pack_exchange(s->d_res, s->n_local, s->global_off, uint64_t(s->lay_x), send, c->stream) != cudaSuccess) {
            c->timer.end(c->stream);
            return fail(c, E2S_ERR_CUDA, "k_pack_exchange");
        }
        if (int rc = cm ? all_gather_rows(c, cm) : E2S_OK) {
            c->timer.end(c->stream);
            return rc;
        }
        MergeParams mp;
        mp.rows = reinterpret_cast<const unsigned long long*>(cm ? cm->d_recv : send);
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
        if (e == cudaSuccess) {
            where = "phase 2 kernels";
            e = snp_run(s->work, a, *p, E2S_MAX_C_LEN, c->d_bases, c->d_off, c->n_reads, c->sm_count, c->stream, &counts, &c->launches, &err,
                        &c->timer, s->d_pf_list, s->pf_cap, &s->d_res->n_pf, &s->d_mout->total.max_clust_length, false);
        }
        if (e == cudaSuccess) {
            where = "copy of the merge result";
            e = cudaMemcpyAsync(&mo, s->d_mout, sizeof mo, cudaMemcpyDeviceToHost, c->stream);
        }
        if (e == cudaSuccess && cm) {
            where = "copy of the exchange rows";
            e = cudaMemcpyAsync(cm->h_recv, cm->d_recv, size_t(world) * XR_WORDS * 8, cudaMemcpyDeviceToHost, c->stream);
        }
        return e == cudaSuccess ? E2S_OK : cuda_fail(c, e, err && err[0] ? err : where);
    };
    // the scan's own synchronisation is the only one of the step
    int rc = run_scan(s, k, min_len, uint32_t(p->mcov_out), true, cm, merge_and_phase2);
    if (rc) return rc;
    const ClusterDev& h = *s->h_pin;
    if (mo.status != MERGE_OK)
        return fail(c, merge_status(mo.status), mo.status == MERGE_EMPTY ? "no clusters (the reference divides by zero here)" : merge_message(mo.status));
    cudaError_t src = cudaSuccess;
    if (!snp_collect(s->work, &counts, &err, &src)) {
        if (src == cudaSuccess)  // a capacity guess of phase 2 was too small: the lists it starts from are still on the device
            src = snp_run(s->work, a, *p, mo.total.max_clust_length, c->d_bases, c->d_off, c->n_reads, c->sm_count, c->stream, &counts,
                          &c->launches, &err, &c->timer, s->d_pf_list, s->pf_cap, &s->d_res->n_pf, nullptr, true);
        if (src == cudaErrorInvalidValue && err && strstr(err, "outside the staged reads")) return fail(c, E2S_ERR_UNSUPPORTED, err);
        if (src != cudaSuccess) return cuda_fail(c, src, err);
    }
    counts.n_analysed = analysed_count(h, mo.mine, p->mcov_out, mo.total.max_clust_length);
    *cnt_out = counts;
    // the shard's state, as e2s_cluster_run + e2s_cluster_finalize + e2s_find_events leave it
    s->rl.scanned(h, uint32_t(p->mcov_out), !s->last_one_pass);
    s->rl.survivors(h.n_pf, true, true);
    s->rl.finalize(mo.mine);
    s->n_variants = cnt_out->n_variants;
    s->events_expanded = false;
    s->rl.events_present(true);
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

// the context's cached resident shard of n positions (the whole eBWT): kept when it has that size, else made anew
static int cached_resident(e2s_ctx* c, uint64_t n, e2s_shard** out) {
    e2s_shard* s = c->cached;
    if (!s || s->chunked || s->n_local != n || s->n_global != n) {
        if (s) e2s_shard_destroy(s);
        c->cached = nullptr;
        if (int rc = e2s_shard_create(c, n, 0, n, &s)) return rc;
        c->cached = s;
    }
    *out = s;
    return E2S_OK;
}

// e2s_pipeline_resident on a sealed resident shard, then its records into rec10 and its events to the caller
static int resident_to_caller(e2s_shard* s, uint32_t k, int32_t min_len, const e2s_snp_params* p, void* rec10, uint64_t cap_records,
                              e2s_event* events, uint64_t cap_events, e2s_pipeline_result* res) {
    int rc;
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

// the same from a resident shard (inputs the one-pass scan does not take: an LCP value above 127, -m > 33)
static int pipeline_host_resident(e2s_ctx* c, const void* gesa, uint64_t n, int x, int y, int z, uint32_t k, int32_t min_len,
                                  const e2s_snp_params* p, void* rec10, uint64_t cap_records, e2s_event* events, uint64_t cap_events,
                                  e2s_pipeline_result* res) {
    int rc;
    e2s_shard* s;
    if ((rc = cached_resident(c, n, &s))) return rc;
    const int rs = x + y + z + 1;
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));  // a cached shard is reloaded from its first position: forget the old verdict
    if ((rc = e2s_shard_load_gesa(s, gesa, 0, n, x, y, z))) return rc;
    if ((rc = e2s_shard_seal(s))) return rc;
    res->h2d_bytes += n * uint64_t(rs);
    return resident_to_caller(s, k, min_len, p, rec10, cap_records, events, cap_events, res);
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

}  // namespace e2s

extern "C" {

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
    // the stream (pipeline_step).
    if (fused_prefilter(p)) {
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

// The sharded step in one call: the resident step of one shard (pipeline_step), the shards' exchange rows all-gathered by
// NCCL on the stream and merged on the device by every rank.  One host synchronisation.
int e2s_pipeline_sharded(e2s_shard* s, e2s_comm* cm, uint32_t k, int32_t min_len, const e2s_snp_params* p, e2s_cluster_merged* mg,
                         e2s_stats* st, e2s_snp_counts* cnt) {
    if (!s || !cm || !p || !mg || !st || !cnt) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_pipeline_sharded: NULL argument");
    if (cm->ctx != s->ctx) return fail(s->ctx, E2S_ERR_ARG, "e2s_pipeline_sharded: communicator belongs to another context");
    return pipeline_step(s, cm, k, min_len, p, mg, st, cnt);
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
    if (min_len > 33 || !fused_prefilter(p))
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

// ebwt2clust + clust2snp from the reads alone: the reads cross PCIe once and serve both the index build (straight into the
// context's resident shard) and phase 2.  Inputs the one-pass scan does not take go where e2s_pipeline_resident sends them.
int e2s_pipeline_reads(e2s_ctx* c, const uint8_t* read_bases, const uint64_t* read_off, uint64_t n_reads, int x, int y, int z, uint32_t k,
                       int32_t min_len, const e2s_snp_params* p, void* rec10, uint64_t cap_records, e2s_event* events, uint64_t cap_events,
                       e2s_pipeline_result* res) {
    if (!c || !read_bases || !read_off || !p || !res) return fail(c, E2S_ERR_ARG, "e2s_pipeline_reads: NULL argument");
    memset(res, 0, sizeof *res);
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, "e2s_pipeline_reads: empty read collection");
    const uint64_t n = read_off[n_reads] + n_reads;
    if ((rc = stage_reads(c, read_bases, read_off, n_reads, res))) return rc;
    e2s_shard* s;
    if ((rc = cached_resident(c, n, &s))) return rc;
    if ((rc = e2s_shard_build_egsa(s, read_off, x, y, z))) return rc;
    if ((rc = e2s_shard_seal(s))) return rc;
    return resident_to_caller(s, k, min_len, p, rec10, cap_records, events, cap_events, res);
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
