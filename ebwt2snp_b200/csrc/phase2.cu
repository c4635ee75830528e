// Phase 2 (clust2snp): statistics() and the exchange between the phases, find_events, and the events out to the caller.

#include <stdlib.h>

#include "host_state.h"
#include "merge.cuh"

using namespace e2s;

namespace e2s {

bool snp_params_ok(const e2s_snp_params* p) {
    return !(p->k_left < 1 || p->k_left > E2S_MAX_K || p->k_right < 1 || p->k_right > E2S_MAX_K || p->max_gap < 1 ||
             p->max_gap > p->k_left || p->max_gap > 255 || p->mcov_out < 1 || 2 * p->mcov_out > E2S_MAX_C_LEN || p->consensus_reads < 1);
}

}  // namespace e2s

extern "C" {

int e2s_statistics(e2s_shard* s, e2s_stats* st) {
    if (!s || !st) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->rl.have_clusters) return fail(c, E2S_ERR_STATE, "no clusters yet");
    CU(c, cudaSetDevice(c->device));
    memset(st, 0, sizeof *st);
    if (!s->rl.staged && s->rl.have_scan_stats) {  // the scan accumulated the histogram of its own records
        for (int i = 0; i < E2S_HIST_BINS; ++i) st->hist[i] = s->rl.h_res.hist[i];
        st->n_bases = s->rl.h_res.n_bases;
        st->n_clust = s->rl.m_own;
        st->last_len = s->rl.h_res.last_rec & 0xffff;
    } else {
    unsigned long long h[E2S_HIST_BINS + 1];
    CU(c, cudaMemsetAsync(s->d_hist, 0, sizeof h, c->stream));
    CU(c, launch_len_hist(s->d_len, s->rl.m_own, s->d_hist, c->stream, c->sm_count));
    ++c->launches;
    CU(c, cudaMemcpyAsync(h, s->d_hist, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    uint16_t last = 0;
    if (s->rl.m_own) CU(c, cudaMemcpyAsync(&last, s->d_len + s->rl.m_own - 1, 2, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < E2S_HIST_BINS; ++i) st->hist[i] = h[i];
    st->n_bases = h[E2S_HIST_BINS];
    st->n_clust = s->rl.m_own;
    st->last_len = last;
    }
    auto add = [&](uint64_t l) {
        if (l <= E2S_MAX_C_LEN) st->hist[l]++;
        st->n_bases += l;
        st->n_clust++;
        st->last_len = l;
    };
    if (!s->rl.staged) {
        if (s->rl.merged.n_prepend && s->rl.merged.prepend_written) {
            const uint64_t keep_last = st->last_len;
            add(s->rl.merged.prepend_len);
            if (s->rl.m_own) st->last_len = keep_last;  // the head record comes first, not last
        }
        for (uint32_t i = 0; i < s->rl.merged.n_append; ++i) add(s->rl.merged.append_len[i]);
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

int e2s_find_events(e2s_shard* s, const e2s_snp_params* p, int max_clust_length, e2s_snp_counts* counts) {
    if (!s || !p || !counts) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    e2s_ctx* c = s->ctx;
    if (!s->rl.have_clusters || !s->rl.finalized) return fail(c, E2S_ERR_STATE, "clusters not computed / staged yet");
    if (!s->sealed) return fail(c, E2S_ERR_STATE, "call e2s_shard_seal after loading the shard");
    if (!c->d_bases) return fail(c, E2S_ERR_STATE, "stage the reads first (e2s_reads_stage)");
    if (!snp_params_ok(p) || max_clust_length > E2S_MAX_C_LEN)
        return fail(c, E2S_ERR_UNSUPPORTED, "clust2snp parameters outside the supported range (DESIGN.md)");
    CU(c, cudaSetDevice(c->device));
    s->rl.events_present(false);
    s->events.clear();
    if (s->rl.staged && s->rl.m_list > 1) {
        // the reference assumes position-ordered, disjoint records (ref:clust2snp.cpp:818-833)
        SnpDev* chk = nullptr;
        CU(c, cudaMalloc(reinterpret_cast<void**>(&chk), sizeof(SnpDev)));
        cudaMemsetAsync(chk, 0, sizeof(SnpDev), c->stream);
        launch_check_sorted(s->d_start, s->d_len, s->rl.m_list, chk, c->stream, c->sm_count);
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
        if (!s->rl.records_flushed || !s->rl.pf_ok || s->rl.pf_mcov != uint32_t(p->mcov_out))
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
            for (int l = 2 * p->mcov_out; l <= max_clust_length; ++l) na0 += s->rl.h_res.hist[l];
            counts->n_analysed = na0;
            s->n_variants = 0;
            s->events_expanded = false;
            s->rl.events_present(true);
            return E2S_OK;
        }
    } else if (!s->rl.staged && s->rl.pf_ok && s->rl.pf_mcov == uint32_t(p->mcov_out) && max_clust_length <= E2S_MAX_C_LEN) {
        SurvEntry extra[4];
        const uint64_t n_extra = s->rl.pf_has_adopted ? 0 : s->rl.merged.n_adopt;  // <= 3 records the merge created and this shard analyses
        for (uint64_t i = 0; i < n_extra && i < 4; ++i)
            extra[i] = SurvEntry{s->rl.merged.adopt_start[i], s->rl.merged.adopt_start[i] - s->global_off, uint32_t(s->rl.merged.adopt_len[i]), 0u};
        if (n_extra) {
            CU(c, cudaMemcpyAsync(s->d_pf_list + s->rl.pf_count, extra, n_extra * sizeof(SurvEntry), cudaMemcpyHostToDevice, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));  // (extra[] lives on this stack frame)
        }
        s->rl.survivors_adopted(n_extra);
        pre_list = s->d_pf_list;
        pre_count = s->rl.pf_count;
    } else {
        int rc = ensure_contiguous(s);  // the two-phase path walks the record list: own records, then the adopted ones
        if (rc) return rc;
        if (!s->rl.staged && s->rl.merged.n_adopt && !s->rl.adopt_put) {
            CU(c, launch_put_records(s->d_start, s->d_len, s->rl.m_own, s->rl.merged.adopt_start, s->rl.merged.adopt_len, int(s->rl.merged.n_adopt), c->stream));
            ++c->launches;
            s->rl.adopted_in_list();
        }
    }
    a.cl_start = s->d_start;
    a.cl_len = s->d_len;
    a.m = s->rl.m_list;
    const char* err = "";
    cudaError_t e = snp_run(s->work, a, *p, max_clust_length, c->d_bases, c->d_off, c->n_reads, c->sm_count, c->stream,
                            counts, &c->launches, &err, &c->timer, pre_list, pre_count);
    if (pre_list && e == cudaSuccess) counts->n_analysed = analysed_count(s->rl.h_res, s->rl.merged, p->mcov_out, max_clust_length);
    if (e == cudaErrorInvalidValue && err && strstr(err, "outside the staged reads")) return fail(c, E2S_ERR_UNSUPPORTED, err);
    if (e != cudaSuccess) return cuda_fail(c, e, err);
    // the packed candidates are already in pinned host memory (K4 wrote them there); they are expanded
    // into e2s_event records when e2s_events_fetch asks for them
    s->n_variants = counts->n_variants;
    s->events_expanded = false;
    s->rl.events_present(true);
    return E2S_OK;
}

int e2s_events_fetch(e2s_shard* s, e2s_event* events, uint64_t cap, uint64_t* n) {
    if (!s || !n) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "NULL argument");
    if (!s->rl.have_events) return fail(s->ctx, E2S_ERR_STATE, "run e2s_find_events first");
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

}  // extern "C"
