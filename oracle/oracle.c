/*
 * oracle.c -- TEST INFRASTRUCTURE ONLY (see oracle.h for the status header).
 *
 * Sequential restatement of the reference algorithm, one function per reference function,
 * each citing the file:line it follows.  Deliberately written as the same state machines the
 * reference runs (NOT as the stencil / scan formulation the CUDA path uses), so that the two
 * are independent derivations checked against each other and against oracle/_ref.
 */
#include "oracle.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define NULLPOS (~(uint64_t)0)

void oracle_default_params(oracle_params *p) {
    p->k_left = 31;
    p->k_right = 30;
    p->mcov_out = 5;
    p->max_gap = 10;
    p->consensus_reads = 20;
    p->max_err = 2;
    p->max_snvs = 3;
    p->pval = 0.99;
    p->nr_reads1 = 0;
}

void oracle_free(void *p) { free(p); }

/* ---- include.hpp helpers ------------------------------------------------------------- */

/* ref:include.hpp:265-279 -- every byte that is not ACGT/acgt (nor N/n) is 0 = 'A' */
static int base_to_int(unsigned char c, uint32_t *flags) {
    switch (c) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    case 'N': case 'n':
        if (flags) *flags |= ORACLE_FLAG_SAW_N; /* reference: rand()%4 -- unpinned */
        return 0;
    default: return 0;
    }
}

/* ref:include.hpp:250-263 */
static unsigned char int_to_base(int i) { return (unsigned char)"ACGT"[i & 3]; }

/* ---- ebwt2clust ----------------------------------------------------------------------- */

/*
 * Value of every 4-byte field of the record "read" after EOF.  The reference's loops are
 * `while(!eof)` over reads that only set eof after failing (ref:ebwt2clust.cpp:90-93,
 * ref:include.hpp:92-107,120-155), so one more record is consumed whose fields are whatever
 * the failed istream::read left in read_el()'s stack locals.  Measured for the oracle/_ref
 * build (g++ 13.3 -Ofast, -x 4 -y 4 -z 4; SURVEY.md §8(a) A3, B2): the low byte is the last
 * byte successfully read (bwt[n-1]) and the upper three bytes are those of the last lcp.
 * ebwt2clust has one exception, handled in oracle_cluster_lm below.
 */
uint32_t oracle_phantom_field(const uint32_t *lcp, const uint8_t *bwt, uint64_t n) {
    return (lcp[n - 1] & 0xFFFFFF00u) | bwt[n - 1];
}

/* ref:ebwt2clust.cpp:54-63 */
static int append_entry(uint64_t *start_out, uint16_t *len_out, uint64_t cap, uint64_t *m, uint64_t start,
                        uint16_t length, int min_len) {
    if ((int)length >= min_len) {
        if (*m >= cap) return -1;
        start_out[*m] = start;
        len_out[*m] = length;
        ++*m;
    }
    return 0;
}

/* ref:ebwt2clust.cpp:68-139 */
int oracle_cluster_lm(const uint32_t *lcp, const uint8_t *bwt, uint64_t n, uint32_t k, int min_len,
                      uint64_t *start_out, uint16_t *len_out, uint64_t cap, oracle_cluster_result *res) {
    return oracle_cluster_lm_x(lcp, bwt, n, k, min_len, 4, start_out, len_out, cap, res);
}

/* Same with the LCP field width of the input file (-x): the failed post-EOF read only touches a temporary of
 * that width (ref:include.hpp:126-155), so the phantom value is the 4-byte rule truncated to lcp_bytes
 * (measured against oracle/_ref for -x 1, 2, 4, 8: tests/test_oracle_golden.py). */
int oracle_cluster_lm_x(const uint32_t *lcp, const uint8_t *bwt, uint64_t n, uint32_t k, int min_len, int lcp_bytes,
                        uint64_t *start_out, uint16_t *len_out, uint64_t cap, oracle_cluster_result *res) {
    const uint32_t pmask = lcp_bytes == 1 ? 0xFFu : (lcp_bytes == 2 ? 0xFFFFu : 0xFFFFFFFFu);
    uint64_t m = 0;
    uint32_t n_clust_out = 0;
    res->n_written = 0;
    res->n_clust_out = 0;
    res->phantom_lcp = 0;
    if (n < 2) return -1; /* the reference reads e1,e2 unconditionally; n<2 is outside its domain */

    uint64_t start;
    uint64_t i;
    uint32_t e1 = lcp[0], e2 = lcp[1], e3;           /* :79-80 */
    start = e1 >= k ? 0 : (e2 >= k ? 1 : NULLPOS);   /* :83-84 */
    i = 1;                                           /* :86 */
    uint64_t next = 2;                               /* next record to read */
    int closed_prev = 0;                             /* did the previous iteration close a cluster */
    uint64_t closed_prev_start = 0;
    int eof = 0;
    while (!eof) {                                   /* :90 */
        if (next < n) {
            e3 = lcp[next++];                        /* :93 */
        } else {
            /* phantom record: stack residue.  If the PREVIOUS iteration closed a cluster (i.e. a
             * cluster ended at index n-2), append_entry's spilled `start` shares the stack slot of
             * the inlined read_el's 4-byte buffer, so the failed read leaves (u32)start there. */
            e3 = (closed_prev ? (uint32_t)closed_prev_start : oracle_phantom_field(lcp, bwt, n)) & pmask;
            res->phantom_lcp = e3;
            eof = 1;
        }
        closed_prev = 0;
        if (start != NULLPOS && ((e1 > e2 && e2 <= e3) || e3 < k)) { /* :98-102 */
            uint16_t length = (uint16_t)((i - start) + 1);            /* :104 */
            if (append_entry(start_out, len_out, cap, &m, start, length, min_len)) return -1;
            n_clust_out++;
            closed_prev = 1;
            closed_prev_start = start;
            start = NULLPOS;
        }
        e1 = e2;                                     /* :112-114 */
        e2 = e3;
        ++i;
        if (start == NULLPOS && e2 >= k) start = i;  /* :116-120 */
    }
    if (start != NULLPOS) {                          /* :127-135 */
        uint16_t length = (uint16_t)((i - start) + 1);
        if (append_entry(start_out, len_out, cap, &m, start, length, min_len)) return -1;
        n_clust_out++;
    }
    res->n_written = m;
    res->n_clust_out = n_clust_out;
    return 0;
}

/* ---- clust2snp: statistics ------------------------------------------------------------ */

/* ref:clust2snp.cpp:877-966 */
int oracle_statistics(const uint64_t *start, const uint16_t *len, uint64_t m, int mcov_out, double pval,
                      oracle_stats *st) {
    (void)start;
    memset(st, 0, sizeof *st);
    if (m == 0) return -1; /* reference: garbage + division by zero */
    const uint64_t MAX_C_LEN = ORACLE_MAX_C_LEN;
    /* while(!eof) { read; ... }: m successful reads + one failed read that leaves the previous
     * (start,length) in place => the last record is processed twice (:889-909) */
    for (uint64_t r = 0; r <= m; ++r) {
        uint16_t length = len[r < m ? r : m - 1];
        if (length <= MAX_C_LEN) {
            st->hist[length]++;
            if (length > st->max_len) st->max_len = length;
        }
        st->n_clust++;
        st->n_bases += length;
    }
    int mcl = 2 * mcov_out;                                        /* :938 */
    if (mcl < 0 || (uint64_t)mcl > MAX_C_LEN) return -1;           /* reference indexes out of bounds */
    uint64_t cumulative = st->hist[mcl] * (uint64_t)mcl;           /* :939 */
    while ((double)cumulative / (double)st->n_bases < pval && (uint64_t)mcl < MAX_C_LEN) { /* :941 */
        mcl++;
        cumulative += st->hist[mcl] * (uint64_t)mcl;
    }
    st->max_clust_length = mcl;
    return 0;
}

/* ---- clust2snp: find_variants --------------------------------------------------------- */

/* A candidate's reads: min(consensus_reads, ORACLE_MAX_C_LEN) per sample at most (an analysed cluster never has more records),
 * so any -c is exact here (the reference keeps them in a vector).  They live in one pool: idx0[n0] pos0[n0] idx1[n1] pos1[n1]
 * from pool[at]. */
typedef struct {
    size_t at; int n0, n1;
    uint64_t right_idx, right_pos;
} candidate;

typedef struct { candidate *v; size_t n, cap; uint64_t *pool; size_t pn, pcap; } cand_vec;

static int cand_push(cand_vec *cv, candidate *c, const uint64_t *idx0, const uint64_t *pos0, const uint64_t *idx1,
                     const uint64_t *pos1) {
    if (cv->n == cv->cap) {
        size_t nc = cv->cap ? cv->cap * 2 : 256;
        candidate *nv = (candidate *)realloc(cv->v, nc * sizeof *nv);
        if (!nv) return -1;
        cv->v = nv;
        cv->cap = nc;
    }
    const size_t need = 2 * (size_t)(c->n0 + c->n1);
    if (cv->pn + need > cv->pcap) {
        size_t nc = cv->pcap ? cv->pcap * 2 : 4096;
        while (nc < cv->pn + need) nc *= 2;
        uint64_t *np = (uint64_t *)realloc(cv->pool, nc * sizeof *np);
        if (!np) return -1;
        cv->pool = np;
        cv->pcap = nc;
    }
    uint64_t *d = cv->pool + cv->pn;
    memcpy(d, idx0, sizeof *d * (size_t)c->n0);
    memcpy(d + c->n0, pos0, sizeof *d * (size_t)c->n0);
    memcpy(d + 2 * c->n0, idx1, sizeof *d * (size_t)c->n1);
    memcpy(d + 2 * c->n0 + c->n1, pos1, sizeof *d * (size_t)c->n1);
    c->at = cv->pn;
    cv->pn += need;
    cv->v[cv->n++] = *c;
    return 0;
}

typedef struct { uint32_t text, suff, lcp; uint8_t bwt; } t_gsa;

/* ref:clust2snp.cpp:367-500 */
static int find_variants(const t_gsa *cl, uint64_t len, const oracle_params *p, cand_vec *out, uint32_t *flags) {
    unsigned counts[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
    uint64_t max_lcp_val = 0, max_idx = 0, max_pos = 0;
    for (uint64_t i = 0; i < len; ++i) {                       /* :377-393 */
        if (cl[i].lcp > max_lcp_val) {
            max_lcp_val = cl[i].lcp;
            max_idx = cl[i].text;
            max_pos = cl[i].suff;
        }
        int sample = cl[i].text < p->nr_reads1 ? 0 : 1;
        counts[sample][base_to_int(cl[i].bwt, flags)]++;
    }
    if (max_lcp_val < (uint64_t)(int64_t)p->k_right) return 0; /* :396 */

    unsigned char f0[4], f1[4];
    int nf0 = 0, nf1 = 0;
    for (int c = 0; c < 4; ++c) {                              /* :402-407, already ascending */
        if (counts[0][c] >= (unsigned)p->mcov_out) f0[nf0++] = int_to_base(c);
        if (counts[1][c] >= (unsigned)p->mcov_out) f1[nf1++] = int_to_base(c);
    }
    int seen[256] = {0}, n_all = 0;                            /* :413-416 */
    for (int a = 0; a < nf0; ++a) if (!seen[f0[a]]++) n_all++;
    for (int a = 0; a < nf1; ++a) if (!seen[f1[a]]++) n_all++;
    int same = nf0 == nf1 && memcmp(f0, f1, (size_t)nf0) == 0;
    if (nf0 == 0 || nf1 == 0 || nf0 > 2 || nf1 > 2 || same || n_all > 3) return 0; /* :419-429 */

    for (int a = 0; a < nf0; ++a) {                            /* :431-496 */
        for (int b = 0; b < nf1; ++b) {
            unsigned char c0 = f0[a], c1 = f1[b];
            if (c0 == c1) continue;
            candidate cd;
            uint64_t idx0[ORACLE_MAX_C_LEN], pos0[ORACLE_MAX_C_LEN], idx1[ORACLE_MAX_C_LEN], pos1[ORACLE_MAX_C_LEN];
            cd.n0 = cd.n1 = 0;
            for (uint64_t i = 0; i < len; ++i) {
                int sample = cl[i].text < p->nr_reads1 ? 0 : 1;
                uint64_t prefix_len = cl[i].suff;
                unsigned char ch = cl[i].bwt;                  /* raw byte compare: '$', 'a' never match */
                uint64_t l = cl[i].lcp;
                if (prefix_len >= (uint64_t)(int64_t)p->k_left && ch == c0 && sample == 0 &&
                    l >= (uint64_t)(int64_t)p->k_right && cd.n0 < p->consensus_reads) {
                    idx0[cd.n0] = cl[i].text;
                    pos0[cd.n0] = cl[i].suff - (uint64_t)p->k_left;
                    cd.n0++;
                }
                if (prefix_len >= (uint64_t)(int64_t)p->k_left && ch == c1 && sample == 1 &&
                    l >= (uint64_t)(int64_t)p->k_right && cd.n1 < p->consensus_reads) {
                    idx1[cd.n1] = cl[i].text;
                    pos1[cd.n1] = cl[i].suff - (uint64_t)p->k_left;
                    cd.n1++;
                }
            }
            if (cd.n0 > 0 && cd.n1 > 0) {
                cd.right_idx = max_idx;
                cd.right_pos = max_pos;
                if (cand_push(out, &cd, idx0, pos0, idx1, pos1)) return -1;
            }
        }
    }
    return 0;
}

/* ---- clust2snp: consensus, distance, output ------------------------------------------ */

/* ref:clust2snp.cpp:218-232 -- right-aligned Hamming distance over the shorter length */
static int dH(const char *a, int la, const char *b, int lb) {
    int len = la < lb ? la : lb, d = 0;
    for (int i = 0; i < len; ++i) d += a[la - i - 1] != b[lb - i - 1];
    return d;
}

/* ref:clust2snp.cpp:254-302 */
void oracle_distance(const char *a, const char *b, int len, int max_gap, int *D, int *gap) {
    int d0 = dH(a, len, b, len);
    if (max_gap == 0) { *D = d0; *gap = 0; return; }
    int min_ab = 0, min_ba = 0, min_ab_idx = 0, min_ba_idx = 0;
    for (int i = 1; i < max_gap + 1; ++i) {                    /* :267-280, first minimum wins */
        int ab = dH(a, len - i, b, len) + i;
        int ba = dH(a, len, b, len - i) + i;
        if (i == 1 || ab < min_ab) { min_ab = ab; min_ab_idx = i - 1; }
        if (i == 1 || ba < min_ba) { min_ba = ba; min_ba_idx = i - 1; }
    }
    if (d0 < min_ab && d0 < min_ba) { *D = d0; *gap = 0; }                          /* :285-288 */
    else if (min_ab < min_ba) { *D = min_ab - (min_ab_idx + 1); *gap = min_ab_idx + 1; } /* :290-294 */
    else { *D = min_ba - (min_ba_idx + 1); *gap = -(min_ba_idx + 1); }              /* :300 */
}

typedef struct { char *s; size_t n, cap; } sbuf;

static int sb_put(sbuf *b, const char *s, size_t n) {
    if (b->n + n + 1 > b->cap) {
        size_t nc = b->cap ? b->cap * 2 : 4096;
        while (nc < b->n + n + 1) nc *= 2;
        char *ns = (char *)realloc(b->s, nc);
        if (!ns) return -1;
        b->s = ns;
        b->cap = nc;
    }
    memcpy(b->s + b->n, s, n);
    b->n += n;
    b->s[b->n] = 0;
    return 0;
}

static int sb_printf_u64(sbuf *b, uint64_t v) {
    char t[32];
    int k = snprintf(t, sizeof t, "%llu", (unsigned long long)v);
    return sb_put(b, t, (size_t)k);
}

/* cons::increment over the listed reads + support count, ref:include.hpp:334-371,
 * ref:clust2snp.cpp:543-593.  Returns -1 on a read reference outside the FASTA. */
static int consensus_support(const uint64_t *idx, const uint64_t *pos, int nr, int k_left, int max_err,
                             const uint8_t *bases, const uint64_t *off, uint64_t n_reads, char *C, int *supp,
                             uint32_t *flags) {
    int cnt[256][4];
    if (k_left > 256) return -1;
    memset(cnt, 0, sizeof(int) * 4 * (size_t)k_left);
    memset(C, 'A', (size_t)k_left);
    for (int j = 0; j < nr; ++j) {
        if (idx[j] >= n_reads || off[idx[j]] + pos[j] + (uint64_t)k_left > off[idx[j] + 1]) {
            *flags |= ORACLE_FLAG_BAD_READ_REF;
            return -1;
        }
        const uint8_t *r = bases + off[idx[j]] + pos[j];
        for (int i = 0; i < k_left; ++i) {
            int b = base_to_int(r[i], flags);
            cnt[i][b]++;
            if (cnt[i][b] > cnt[i][base_to_int((unsigned char)C[i], flags)]) C[i] = (char)r[i];
        }
    }
    *supp = 0;
    for (int j = 0; j < nr; ++j) {
        const uint8_t *r = bases + off[idx[j]] + pos[j];
        int d = 0;
        for (int i = 0; i < k_left; ++i) d += C[i] != (char)r[i];
        if (d <= max_err) ++*supp;
    }
    return 0;
}

/* one event, ref:clust2snp.cpp:644-766 */
static int emit_event(sbuf *o, uint64_t id_nr, const char *l0, const char *l1, int kl, const char *right, int rl,
                      int supp0, int supp1, int gap) {
    char type[300];
    int tn = 0;
    if (gap == 0) { type[tn++] = l0[kl - 1]; type[tn++] = '/'; type[tn++] = l1[kl - 1]; }
    else if (gap > 0) { memcpy(type, l0 + kl - gap, (size_t)gap); tn = gap; type[tn++] = '/'; }
    else { type[tn++] = '/'; memcpy(type + tn, l1 + kl - (-gap), (size_t)(-gap)); tn += -gap; }
    for (int path = 0; path < 2; ++path) {
        const char *hdr = gap != 0 ? (path ? ">INDEL_lower_path_" : ">INDEL_higher_path_")
                                   : (path ? ">SNP_lower_path_" : ">SNP_higher_path_");
        if (sb_put(o, hdr, strlen(hdr)) || sb_printf_u64(o, id_nr) || sb_put(o, "|P_1:", 5) ||
            sb_printf_u64(o, (uint64_t)rl) || sb_put(o, "_", 1) || sb_put(o, type, (size_t)tn) || sb_put(o, "|", 1) ||
            sb_printf_u64(o, (uint64_t)(path ? supp1 : supp0)) || sb_put(o, "|nb_pol_1\n", 10))
            return -1;
        const char *l = path ? l1 : l0;
        int skip = 0;
        if (path == 0 && gap < 0) skip = -gap;   /* :711 */
        if (path == 1 && gap > 0) skip = gap;    /* :753 */
        if (sb_put(o, l + skip, (size_t)(kl - skip)) || sb_put(o, right, (size_t)rl) || sb_put(o, "\n", 1)) return -1;
    }
    return 0;
}

/* The record "read" after EOF (SURVEY.md 8(a) A3/B2), for any field widths.  read_el's four temporaries
 * (ref:include.hpp:126-155 / :159-188) share one 8-byte stack slot; a failed read leaves it untouched, so the
 * phantom field of width w is the low w bytes of what the LAST VALID record left there: byte 0 = bwt[n-1]
 * (read last), byte b >= 1 = byte b of the last-read field that is wider than b -- lcp, then (EGSA order
 * text, suff, lcp) suff, then text; in BCR order (suff, text, lcp) text before suff.  Measured against
 * oracle/_ref by bisection on -n for ten width combinations in both file formats (tests/golden/make_golden.py,
 * phantom_tail cases). */
uint64_t oracle_phantom_slot(uint32_t lcp_last, uint32_t text_last, uint32_t suff_last, uint8_t bwt_last,
                             int x, int y, int z, int bcr) {
    uint64_t slot = bwt_last;
    for (int b = 1; b < 8; ++b) {
        uint64_t v = 0; /* 8-byte fields: bytes 4..7 of the file value are not kept by this restatement (always 0 here) */
        if (b < x) v = b < 4 ? (lcp_last >> (8 * b)) & 0xff : 0;
        else if (!bcr && b < z) v = b < 4 ? (suff_last >> (8 * b)) & 0xff : 0;
        else if (b < y) v = b < 4 ? (text_last >> (8 * b)) & 0xff : 0;
        else if (bcr && b < z) v = b < 4 ? (suff_last >> (8 * b)) & 0xff : 0;
        slot |= v << (8 * b);
    }
    return slot;
}
static uint32_t slot_field(uint64_t slot, int w) {
    return (uint32_t)(w >= 4 ? slot : slot & ((1ull << (8 * w)) - 1));
}

int oracle_find_events(const uint32_t *lcp, const uint32_t *text, const uint32_t *suff, const uint8_t *bwt,
                       uint64_t n, const uint64_t *start, const uint16_t *len, uint64_t m,
                       const oracle_params *p, int max_clust_length,
                       const uint8_t *read_bases, const uint64_t *read_off, uint64_t n_reads,
                       char **snp_text, size_t *snp_len, oracle_snp_result *res) {
    return oracle_find_events_w(lcp, text, suff, bwt, n, start, len, m, p, max_clust_length, read_bases, read_off, n_reads,
                                4, 4, 4, 0, snp_text, snp_len, res);
}

/* ref:clust2snp.cpp:788-872 (find_events), :505-628 (extract_variants), :633-780 (to_file); x, y, z = byte widths of
 * lcp / text / suff in the index files, bcr = 1 for the BCR triple (they only matter for the phantom record) */
int oracle_find_events_w(const uint32_t *lcp, const uint32_t *text, const uint32_t *suff, const uint8_t *bwt,
                         uint64_t n, const uint64_t *start, const uint16_t *len, uint64_t m,
                         const oracle_params *p, int max_clust_length,
                         const uint8_t *read_bases, const uint64_t *read_off, uint64_t n_reads,
                         int x, int y, int z, int bcr,
                         char **snp_text, size_t *snp_len, oracle_snp_result *res) {
    memset(res, 0, sizeof *res);
    *snp_text = NULL;
    *snp_len = 0;
    /* outside what this restatement supports (an empty index, -c < 1, -L > 256, -g > -L, clusters longer than the reference's
     * MAX_C_LEN): refused, with no flag set */
    if (n == 0 || p->consensus_reads < 1 || p->k_left > 256 || p->max_gap > p->k_left || max_clust_length > ORACLE_MAX_C_LEN)
        return -1;
    cand_vec cands = {0, 0, 0, 0, 0, 0};
    t_gsa *cl = (t_gsa *)malloc(65536 * sizeof *cl);
    if (!cl) return -1;
    const uint64_t slot = oracle_phantom_slot(lcp[n - 1], text[n - 1], suff[n - 1], bwt[n - 1], x, y, z, bcr);
    int rc = 0;

    /* forward-only cursor over the EGSA; `e` is always record i (the phantom one for i >= n) */
    uint64_t i = 0;
    for (uint64_t r = 0; r <= m && !rc; ++r) {       /* m records + the duplicated last one (:806) */
        uint64_t st = start[r < m ? r : m - 1];
        uint16_t length = len[r < m ? r : m - 1];
        if ((int)length >= p->mcov_out * 2 && (int)length <= max_clust_length) { /* :816 */
            while (i < st) ++i;                      /* :818-823 */
            uint64_t cnt = 0;
            while (i < st + length) {                /* :827-833 */
                t_gsa e;
                if (i < n) { e.text = text[i]; e.suff = suff[i]; e.lcp = lcp[i]; e.bwt = bwt[i]; }
                else {
                    e.text = slot_field(slot, y);
                    e.suff = slot_field(slot, z);
                    e.lcp = slot_field(slot, x);
                    e.bwt = bwt[n - 1];
                }
                cl[cnt++] = e;
                ++i;
            }
            if (r < m) res->n_analysed++;
            rc = find_variants(cl, cnt, p, &cands, &res->flags); /* :840-843 */
        }
    }
    free(cl);
    res->n_candidates = cands.n;

    /* extract_variants + to_file fused: per candidate, in order */
    sbuf out = {0, 0, 0};
    if (!rc && sb_put(&out, "", 0)) rc = -1;
    uint64_t id_nr = 1;
    char l0[256], l1[256];
    for (size_t c = 0; c < cands.n && !rc; ++c) {
        const candidate *v = &cands.v[c];
        const uint64_t *r0 = cands.pool + v->at, *r1 = r0 + 2 * v->n0;
        int supp0 = 0, supp1 = 0;
        if (consensus_support(r0, r0 + v->n0, v->n0, p->k_left, p->max_err, read_bases, read_off, n_reads, l0,
                              &supp0, &res->flags) ||
            consensus_support(r1, r1 + v->n1, v->n1, p->k_left, p->max_err, read_bases, read_off, n_reads, l1,
                              &supp1, &res->flags)) { rc = -1; break; }
        if (!(supp0 > 0 && supp1 > 0)) continue;     /* :595 */
        if (v->right_idx >= n_reads) { res->flags |= ORACLE_FLAG_BAD_READ_REF; rc = -1; break; }
        uint64_t rlen = read_off[v->right_idx + 1] - read_off[v->right_idx];
        if (v->right_pos > rlen) { res->flags |= ORACLE_FLAG_BAD_READ_REF; rc = -1; break; } /* substr throws */
        uint64_t rl = rlen - v->right_pos;           /* substr clamps (:604) */
        if (rl > (uint64_t)p->k_right) rl = (uint64_t)p->k_right;
        const char *right = (const char *)read_bases + read_off[v->right_idx] + v->right_pos;
        res->n_variants++;
        int D, gap;
        oracle_distance(l0, l1, p->k_left, p->max_gap, &D, &gap);
        if (D <= p->max_snvs) {                      /* :648 */
            if (emit_event(&out, id_nr, l0, l1, p->k_left, right, (int)rl, supp0, supp1, gap)) { rc = -1; break; }
            id_nr++;
            res->n_events++;
        }
    }
    free(cands.v);
    free(cands.pool);
    if (rc) { free(out.s); return -1; }
    *snp_text = out.s;
    *snp_len = out.n;
    return 0;
}


/* ------------------------------------------------------------------------------------------
 * EGSA construction (SURVEY.md 8(f) rank 1).  PARITY UNPINNED against the real thing: the reference delegates this step
 * to the external `egsa` / BCR programs (ref:README.md:46-60, ref:pipeline.sh:98-109), which are neither vendored in
 * /root/reference nor installed here, and nothing in the reference tree pins their terminator byte or tie order
 * (SURVEY.md 8(b), last row).  This is the textbook definition -- sort all suffixes of all reads, `$` < A < C < G < T,
 * equal suffixes by read id -- written as a comparison sort over (read, offset) pairs, with the conventions this
 * repository's synthetic data has always used (ebwt2snp_b200/synth.py).  It checks the CUDA builder (e2s_build_egsa_dev).
 * ------------------------------------------------------------------------------------------ */
#include <stdlib.h>

static const uint8_t *g_sort_reads;
static uint32_t g_sort_L;

static int suffix_cmp(const void *pa, const void *pb) {
    const uint64_t a = *(const uint64_t *)pa, b = *(const uint64_t *)pb;
    const uint64_t ra = a / (g_sort_L + 1), rb = b / (g_sort_L + 1);
    const uint32_t oa = (uint32_t)(a % (g_sort_L + 1)), ob = (uint32_t)(b % (g_sort_L + 1));
    const uint8_t *sa = g_sort_reads + ra * g_sort_L + oa, *sb = g_sort_reads + rb * g_sort_L + ob;
    const uint32_t la = g_sort_L - oa, lb = g_sort_L - ob, lm = la < lb ? la : lb;
    for (uint32_t i = 0; i < lm; ++i) {
        if (sa[i] != sb[i]) return sa[i] < sb[i] ? -1 : 1; /* ASCII order of ACGT = code order */
    }
    if (la != lb) return la < lb ? -1 : 1; /* the terminator is smaller than every base */
    return ra < rb ? -1 : (ra > rb ? 1 : 0);
}

int oracle_build_egsa(const uint8_t *reads, uint64_t n_reads, uint32_t read_len, uint32_t *lcp, uint32_t *text,
                      uint32_t *suff, uint8_t *bwt) {
    const uint64_t n = n_reads * ((uint64_t)read_len + 1);
    uint64_t *idx = (uint64_t *)malloc(n * sizeof *idx);
    if (!idx) return -1;
    for (uint64_t i = 0; i < n; ++i) idx[i] = i;
    g_sort_reads = reads;
    g_sort_L = read_len;
    qsort(idx, n, sizeof *idx, suffix_cmp);
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t r = idx[i] / (read_len + 1);
        const uint32_t o = (uint32_t)(idx[i] % (read_len + 1));
        text[i] = (uint32_t)r;
        suff[i] = o;
        bwt[i] = o ? reads[r * read_len + o - 1] : (uint8_t)'$';
        uint32_t l = 0;
        if (i) {
            const uint64_t r0 = idx[i - 1] / (read_len + 1);
            const uint32_t o0 = (uint32_t)(idx[i - 1] % (read_len + 1));
            const uint32_t lm = read_len - (o0 > o ? o0 : o);
            while (l < lm && reads[r0 * read_len + o0 + l] == reads[r * read_len + o + l]) ++l;
        }
        lcp[i] = l;
    }
    free(idx);
    return 0;
}

/* The same for reads of any lengths (the reference's FASTA parser accepts them, ref:clust2snp.cpp:147-212; empty reads
 * included): bases = all reads back to back, off = n_reads + 1 offsets.  n = off[n_reads] + n_reads records.
 * Checks e2s_build_egsa_ragged(_dev).  A suffix is (read << 32 | offset). */
static const uint64_t *g_sort_off;

static int ragged_cmp(const void *pa, const void *pb) {
    const uint64_t a = *(const uint64_t *)pa, b = *(const uint64_t *)pb;
    const uint64_t ra = a >> 32, rb = b >> 32;
    const uint32_t oa = (uint32_t)a, ob = (uint32_t)b;
    const uint8_t *sa = g_sort_reads + g_sort_off[ra] + oa, *sb = g_sort_reads + g_sort_off[rb] + ob;
    const uint32_t la = (uint32_t)(g_sort_off[ra + 1] - g_sort_off[ra]) - oa, lb = (uint32_t)(g_sort_off[rb + 1] - g_sort_off[rb]) - ob;
    const uint32_t lm = la < lb ? la : lb;
    for (uint32_t i = 0; i < lm; ++i) {
        if (sa[i] != sb[i]) return sa[i] < sb[i] ? -1 : 1;
    }
    if (la != lb) return la < lb ? -1 : 1;
    return ra < rb ? -1 : (ra > rb ? 1 : 0);
}

int oracle_build_egsa_ragged(const uint8_t *bases, const uint64_t *off, uint64_t n_reads, uint32_t *lcp, uint32_t *text,
                             uint32_t *suff, uint8_t *bwt) {
    const uint64_t n = off[n_reads] + n_reads;
    uint64_t *idx = (uint64_t *)malloc((n ? n : 1) * sizeof *idx);
    if (!idx) return -1;
    uint64_t at = 0;
    for (uint64_t r = 0; r < n_reads; ++r)
        for (uint64_t o = 0; o <= off[r + 1] - off[r]; ++o) idx[at++] = (r << 32) | o;
    g_sort_reads = bases;
    g_sort_off = off;
    qsort(idx, n, sizeof *idx, ragged_cmp);
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t r = idx[i] >> 32;
        const uint32_t o = (uint32_t)idx[i];
        text[i] = (uint32_t)r;
        suff[i] = o;
        bwt[i] = o ? bases[off[r] + o - 1] : (uint8_t)'$';
        uint32_t l = 0;
        if (i) {
            const uint64_t r0 = idx[i - 1] >> 32;
            const uint32_t o0 = (uint32_t)idx[i - 1];
            const uint32_t la = (uint32_t)(off[r + 1] - off[r]) - o, lb = (uint32_t)(off[r0 + 1] - off[r0]) - o0;
            const uint32_t lm = la < lb ? la : lb;
            while (l < lm && bases[off[r0] + o0 + l] == bases[off[r] + o + l]) ++l;
        }
        lcp[i] = l;
    }
    free(idx);
    return 0;
}
