// The integer logic between the two phases, written once for host and device: chaining the shards' open-cluster states,
// the tail + post-EOF phantom rule of cluster_lm (ref:ebwt2clust.cpp:90-135; SURVEY.md 8(a) A3) and the pval loop of
// statistics() (ref:clust2snp.cpp:889-946).  The C ABI entry points (e2s_cluster_merge, e2s_statistics_finish,
// e2s_exchange_finish: phase1.cu, phase2.cu) wrap these on the host; k_merge_stats runs the same code in one thread on the device, so
// that a resident step never leaves the stream between the scan and phase 2.
#pragma once

#include <stdint.h>

#include "../../include/ebwt2snp_b200.h"

#ifdef __CUDACC__
#define E2S_HD __host__ __device__
#else
#define E2S_HD
#endif

namespace e2s {

enum { MERGE_OK = 0, MERGE_NOT_PARTITION = 1, MERGE_NOT_COVER = 2, MERGE_END_WITHOUT_START = 3, MERGE_EMPTY = 4, MERGE_BAD_MCOV = 5 };

// e2s_cluster_merge: the view of shard `my` after all shards' summaries have been chained
E2S_HD inline int merge_core(const e2s_cluster_summary* all, int n_shards, int my, e2s_cluster_merged* out) {
    *out = e2s_cluster_merged{};
    const uint64_t n = all[0].n_global;
    const uint32_t k = uint32_t(all[0].k);
    const int64_t min_len = int64_t(all[0].min_len);
    uint64_t expect = 0;
    for (int g = 0; g < n_shards; ++g) {
        if (all[g].global_off != expect || all[g].n_global != n || all[g].k != all[0].k || all[g].min_len != all[0].min_len)
            return MERGE_NOT_PARTITION;
        expect += all[g].n_local;
    }
    if (expect != n) return MERGE_NOT_COVER;
    auto owner = [&](uint64_t pos) {
        for (int g = 0; g < n_shards; ++g)
            if (pos < all[g].global_off + all[g].n_local) return g;
        return n_shards - 1;  // position n (phantom-only cluster) stays with the last shard
    };
    auto adopt = [&](uint64_t st, uint64_t len) {
        if (owner(st) == my && out->n_adopt < 3) {
            out->adopt_start[out->n_adopt] = st;
            out->adopt_len[out->n_adopt] = len;
            out->n_adopt++;
        }
    };
    uint64_t s_open = 0;  // 1 + global start of the open cluster, 0 = none
    uint64_t offset = 0, closed = 0;
    uint64_t last_head_start = 0;
    for (int g = 0; g < n_shards; ++g) {
        if (g == my) out->record_offset = offset;
        if (all[g].head_end) {
            if (!s_open) return MERGE_END_WITHOUT_START;
            const uint64_t st = s_open - 1, en = all[g].head_end - 1;
            const uint64_t len = (en - st + 1) & 0xffff;
            const bool written = int64_t(len) >= min_len;
            if (g == my) {
                out->n_prepend = 1;
                out->prepend_start = st;
                out->prepend_len = len;
                out->prepend_written = written;
            }
            if (written) {
                offset += 1;
                adopt(st, len);
            }
            last_head_start = st;
            s_open = 0;
        }
        offset += all[g].n_written;
        closed += all[g].n_end;
        if (all[g].any_event) s_open = all[g].open_start;
    }
    // tail: position n-1 with the phantom record as its right neighbour, then position n
    const e2s_cluster_summary& L = all[n_shards - 1];
    const uint32_t e1 = uint32_t(L.tail_lcp_nm2), e2 = uint32_t(L.tail_lcp_nm1);
    uint32_t P;
    if (L.end_nm2_start == ~0ull) P = uint32_t(last_head_start);
    else if (L.end_nm2_start) P = uint32_t(L.end_nm2_start - 1);
    else P = (e2 & 0xFFFFFF00u) | uint32_t(L.tail_bwt_nm1 & 0xff);
    // the failed read only touches a temporary of the LCP field's width (ref:include.hpp:126-155)
    if (L.lcp_bytes == 1) P &= 0xFFu;
    else if (L.lcp_bytes == 2) P &= 0xFFFFu;
    out->phantom_lcp = P;
    uint32_t na = 0;
    auto tail_record = [&](uint64_t st, uint64_t en) {
        const uint64_t len = (en - st + 1) & 0xffff;
        ++closed;
        if (int64_t(len) >= min_len) {
            offset += 1;
            if (my == n_shards - 1) {
                out->append_start[na] = st;
                out->append_len[na] = len;
                ++na;
            }
            adopt(st, len);
        }
    };
    if (s_open && ((e1 > e2 && e2 <= P) || P < k)) {
        tail_record(s_open - 1, n - 1);
        s_open = 0;
    }
    if (!s_open && P >= k) s_open = n + 1;
    if (s_open) tail_record(s_open - 1, n);
    out->n_append = na;
    out->total_written = offset;
    out->n_clust_out = closed;
    return MERGE_OK;
}

// e2s_statistics_finish: the reference counts the last record twice, then runs the pval loop -- one IEEE double division
// per step (ref:clust2snp.cpp:938-946; the device's division is the same correctly rounded operation)
// first half (serial, cheap): the double-counted last record, max_len, the mcov check
E2S_HD inline int stats_finish_head(e2s_stats* st, uint64_t last_len, int mcov_out) {
    if (st->n_clust == 0) return MERGE_EMPTY;
    if (last_len <= E2S_MAX_C_LEN) st->hist[last_len]++;
    st->n_clust++;
    st->n_bases += last_len;
    st->max_len = 0;
    for (int i = 0; i < E2S_HIST_BINS; ++i)
        if (st->hist[i]) st->max_len = uint64_t(i);
    const int mcl = 2 * mcov_out;
    if (mcl < 0 || mcl > E2S_MAX_C_LEN) return MERGE_BAD_MCOV;
    return MERGE_OK;
}

E2S_HD inline int stats_finish_core(e2s_stats* st, uint64_t last_len, int mcov_out, double pval) {
    const int rc = stats_finish_head(st, last_len, mcov_out);
    if (rc != MERGE_OK) return rc;
    int mcl = 2 * mcov_out;
    uint64_t cumulative = st->hist[mcl] * uint64_t(mcl);
    while (double(cumulative) / double(st->n_bases) < pval && mcl < E2S_MAX_C_LEN) {
        mcl++;
        cumulative += st->hist[mcl] * uint64_t(mcl);
    }
    st->max_clust_length = mcl;
    return MERGE_OK;
}

}  // namespace e2s
