/*
 * ebwt2snp_b200.h -- C ABI of the B200 (sm_100a) implementation of the ebwt2snp hot path:
 * ebwt2clust's eBWT/LCP scan into positional clusters and clust2snp's per-cluster SNP/indel
 * calling (reference: nicolaprezza/ebwt2snp; `ref:` citations are file:line in that tree).
 *
 * The reference exposes no plugin / FFI interface: its contract for this path is the process
 * boundary of the two CLIs (argv + files).  This header is the thin layer between those CLIs
 * (re-implemented in ebwt2snp_b200/host/) and the CUDA kernels; each entry point names the
 * reference function whose work it takes over.  INTEGRATION.md shows the binding a maintainer
 * of the reference would add to call it from ebwt2clust.cpp / clust2snp.cpp.
 *
 * Conventions: plain C types, caller-owned host buffers, int status return (0 = E2S_OK),
 * no exceptions cross the boundary, no torch types.  A context is bound to one CUDA device
 * and one stream; calls on one context are not thread-safe.  There is NO CPU fallback:
 * every compute entry point fails with E2S_ERR_CUDA when no sm_100 device is usable.
 *
 * Positions are eBWT positions (= EGSA records).  A *shard* is a contiguous range
 * [global_off, global_off + n_local) of the n_global positions, resident in HBM as
 * structure-of-arrays (lcp u32, text u32, suff u32, bwt u8) with the halos the kernels need
 * (2 left / 1 right LCP values for the cluster flags, E2S_MAX_C_LEN records on the right for
 * the per-cluster analysis).  One GPU holds one shard at a time; multi-GPU = one shard per
 * GPU (or per process) plus e2s_cluster_merge() on the all-gathered summaries.
 */
#ifndef EBWT2SNP_B200_H
#define EBWT2SNP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define E2S_VERSION 100

/* status codes */
#define E2S_OK 0
#define E2S_ERR_CUDA 1        /* CUDA runtime error / no device (message in e2s_last_error) */
#define E2S_ERR_ARG 2         /* invalid argument */
#define E2S_ERR_NOMEM 3       /* host or device allocation failed */
#define E2S_ERR_UNSUPPORTED 4 /* input outside the supported domain (documented in DESIGN.md) */
#define E2S_ERR_STATE 5       /* call sequence error (e.g. clusters not computed yet) */

#define E2S_MAX_C_LEN 150 /* ref:clust2snp.cpp:32  max_clust_length_def (the -M option is unreachable) */
#define E2S_MAX_K 128     /* largest -L / -R context length supported by the event records */
#define E2S_HIST_BINS (E2S_MAX_C_LEN + 1)

typedef struct e2s_ctx e2s_ctx;
typedef struct e2s_shard e2s_shard;
typedef struct e2s_comm e2s_comm; /* one process per GPU: wraps an NCCL communicator (e2s_comm_create), or the caller's own
                                     all-gather (e2s_comm_create_gather: several ranks on one GPU, as the tests run them) */

/* ---------------------------------------------------------------------------------------
 * context
 * ------------------------------------------------------------------------------------- */
int e2s_version(void);
/* E2S_SM_COUNT=s in the environment (a test hook, 1 <= s <= the device's SM count, else E2S_ERR_ARG) sizes every grid of
 * the context for s SMs, so that CTAs loop over many tiles and grid-stride rounds at small inputs. */
int e2s_ctx_create(int device, e2s_ctx **out);
void e2s_ctx_destroy(e2s_ctx *ctx);
/* last error message of the context (or of the calling thread when ctx == NULL) */
const char *e2s_last_error(const e2s_ctx *ctx);
/* use an existing CUDA stream (cudaStream_t passed as void*) instead of the context's own */
int e2s_ctx_set_stream(e2s_ctx *ctx, void *cuda_stream);
int e2s_ctx_synchronize(e2s_ctx *ctx);
/* free / total device memory of the context's GPU right now (the CLIs choose between a resident and a chunked shard with it) */
int e2s_ctx_mem_info(e2s_ctx *ctx, uint64_t *free_bytes, uint64_t *total_bytes);
/* the CUDA devices this process sees */
int e2s_device_count(int *count);
/* number of kernel launches issued through this context so far (bench.py's gpu_launches) */
uint64_t e2s_ctx_launch_count(const e2s_ctx *ctx);
/* Per-kernel device time, measured with CUDA events recorded on the context's stream around the
 * kernels that touch every position (bench.py's roofline).  e2s_ctx_kernel_time synchronises
 * the stream, returns the time and launch count accumulated since the last call and resets them. */
#define E2S_KERNEL_FLAGS 0 /* K1: LCP boundary stencil -> START/END bit masks */
#define E2S_KERNEL_EMIT 1  /* K2: look-back scan over the masks + record compaction */
#define E2S_KERNEL_SCAN 2  /* K3a: per-cluster base-code prefilter on the resident bit planes of the BWT */
#define E2S_KERNEL_EXACT 3 /* K3x: exact 2x4 histogram / filters of the surviving clusters */
#define E2S_KERNEL_SCAN1 4 /* K1 + K2 in one pass over the bit-sliced LCP (k_cluster_scan): what runs whenever the shard has it */
#define E2S_KERNEL_RESOLVE 5 /* k_chunk_resolve: chunk heads, segment offsets, shard totals */
#define E2S_KERNEL_CAND 6   /* K3b: candidate slots of the flagged clusters */
#define E2S_KERNEL_EVENTS 7 /* K4: contexts, consensus, support, distance, event records to pinned host memory */
#define E2S_KERNEL_MERGE 8  /* k_pack_exchange [+ ncclAllGather] + k_merge_stats: the exchange between the phases (pipelines only) */
#define E2S_KERNEL_COUNT 9
int e2s_ctx_timing(e2s_ctx *ctx, int enable);
int e2s_ctx_kernel_time(e2s_ctx *ctx, int kernel, double *total_ms, uint64_t *launches);

/* ---------------------------------------------------------------------------------------
 * shard residency  (replaces egsa_stream: ref:include.hpp:32-219)
 * ------------------------------------------------------------------------------------- */
int e2s_shard_create(e2s_ctx *ctx, uint64_t n_local, uint64_t global_off, uint64_t n_global, e2s_shard **out);
void e2s_shard_destroy(e2s_shard *sh);

/* Host array-of-structs EGSA records exactly as in X.gesa: text(y) suff(z) lcp(x) bwt(1),
 * little endian, x,y,z in {1,2,4,8} (values wider than 32 bits truncated as ref:include.hpp:131,140,149).
 * `records` holds `count` records, the first being global position `first`.  May be called
 * repeatedly with consecutive chunks; the shard keeps what falls in
 * [global_off - 2, global_off + n_local + E2S_MAX_C_LEN + 1) and ignores the rest.
 * The copy is H2D of the raw bytes followed by a de-interleave kernel. */
int e2s_shard_load_gesa(e2s_shard *sh, const void *records, uint64_t first, uint64_t count, int x, int y, int z);
/* The same straight from an open X.gesa file (record i at byte i * (x + y + z + 1) = global position i): what egsa_stream does
 * with one istream::read per field (ref:include.hpp:42-81,120-155).  Reader threads (E2S_READ_THREADS, default 6) pread()
 * pieces into a pinned ring while earlier pieces are copied and de-interleaved. */
int e2s_shard_load_gesa_fd(e2s_shard *sh, int fd, uint64_t first, uint64_t count, int x, int y, int z);

/* Host structure-of-arrays (BCR-like: ref:include.hpp:157-188).  Arrays may be NULL to skip a field. */
int e2s_shard_load_soa(e2s_shard *sh, const uint32_t *lcp, const uint32_t *text, const uint32_t *suff,
                       const uint8_t *bwt, uint64_t first, uint64_t count);
/* Same, from DEVICE pointers on the context's device (device-to-device copies). */
int e2s_shard_load_soa_dev(e2s_shard *sh, const uint32_t *d_lcp, const uint32_t *d_text, const uint32_t *d_suff,
                           const uint8_t *d_bwt, uint64_t first, uint64_t count);
/* EGSA construction on the GPU (SURVEY.md 8(f) rank 1): what the reference expects an external egsa / BCR run to have
 * produced before either tool starts (ref:README.md:46-60, ref:pipeline.sh:98-109).  Suffix-sorts a collection of
 * n_reads reads of read_len ACGT bases each (DEVICE pointer, row-major ASCII, no separators) and writes the four arrays
 * of n = n_reads * (read_len + 1) records to DEVICE memory, ready for e2s_shard_load_soa_dev: one record per suffix
 * incl. the terminator suffix, `$` < A < C < G < T, equal suffixes by read id, lcp never extends over a terminator,
 * bwt = preceding base or `$` (0x24).  The sort is the library's own radix sort (csrc/build_egsa.cu); suffix ids are
 * 32-bit while n < 2^32 and 64-bit beyond (scratch: 24.5 / 32.5 bytes per suffix).  Synchronises the context's stream. */
int e2s_build_egsa_dev(e2s_ctx *ctx, const uint8_t *d_reads, uint64_t n_reads, uint32_t read_len, uint32_t *d_lcp,
                       uint32_t *d_text, uint32_t *d_suff, uint8_t *d_bwt);

/* Same from / to HOST memory (what ebwt2snp_b200/bin/build_gesa uses): device buffers are allocated and released inside. */
int e2s_build_egsa(e2s_ctx *ctx, const uint8_t *reads, uint64_t n_reads, uint32_t read_len, uint32_t *lcp, uint32_t *text,
                   uint32_t *suff, uint8_t *bwt);

/* Reads of ANY lengths, as the reference's FASTA parser accepts them (ref:clust2snp.cpp:147-212; empty reads included):
 * d_bases = all reads back to back (DEVICE pointer), off = n_reads + 1 offsets into it in HOST memory (off[0] = 0,
 * non-decreasing, every read shorter than 65536 bases).  n = off[n_reads] + n_reads records, same conventions. */
int e2s_build_egsa_ragged_dev(e2s_ctx *ctx, const uint8_t *d_bases, const uint64_t *off, uint64_t n_reads, uint32_t *d_lcp,
                              uint32_t *d_text, uint32_t *d_suff, uint8_t *d_bwt);
int e2s_build_egsa_ragged(e2s_ctx *ctx, const uint8_t *bases, const uint64_t *off, uint64_t n_reads, uint32_t *lcp,
                          uint32_t *text, uint32_t *suff, uint8_t *bwt);

/* ONE KEY RANGE of the index of n_reads equal-length reads (any lengths: e2s_build_egsa_ragged_range_dev below): the suffixes whose first 32 symbols -- as a 64-bit word at 2 bits per
 * base (A=0 C=1 G=2 T=3, first symbol most significant, zero padded past the end of the read) -- lie in [key_lo, key_hi)
 * (key_hi = 0: no upper bound) are a contiguous range of the index.  Writes their records to the DEVICE arrays (capacity
 * records each), *n_records = how many, *first_position = the index position of the first one.  What a collection too large for one
 * call's scratch is built from (range after range on one GPU), and what each GPU of a box builds for its shard (the egsa / BCR run
 * of ref:pipeline.sh:98-109 sharded by key).  (before_text, before_suff) = the record that precedes the range, for lcp[0];
 * before_text = 0xFFFFFFFF: none / not known, lcp[0] = 0.  More records than capacity: E2S_ERR_ARG, nothing written, *n_records set.
 * Scratch: 24.5 / 32.5 bytes per suffix of the RANGE.  Synchronises the context's stream. */
int e2s_build_egsa_range_dev(e2s_ctx *ctx, const uint8_t *d_reads, uint64_t n_reads, uint32_t read_len, uint64_t key_lo,
                             uint64_t key_hi, uint32_t before_text, uint32_t before_suff, uint64_t capacity, uint32_t *d_lcp,
                             uint32_t *d_text, uint32_t *d_suff, uint8_t *d_bwt, uint64_t *n_records, uint64_t *first_position);

/* The same for reads of ANY lengths: d_bases / off as for e2s_build_egsa_ragged_dev (off = n_reads + 1 HOST offsets, checked the
 * same way).  The suffix ids follow the whole collection (64-bit when n_reads << bits(longest read + 1) exceeds 2^32), so the ranges of
 * one collection concatenate to exactly the index e2s_build_egsa_ragged_dev writes.  Capacity, before and errors as above; a base
 * outside ACGT or a read of 65536 bases or more: E2S_ERR_UNSUPPORTED.  e2s_build_egsa_ragged switches to these ranges by itself when
 * the whole index does not fit the device. */
int e2s_build_egsa_ragged_range_dev(e2s_ctx *ctx, const uint8_t *d_bases, const uint64_t *off, uint64_t n_reads, uint64_t key_lo,
                                    uint64_t key_hi, uint32_t before_text, uint32_t before_suff, uint64_t capacity, uint32_t *d_lcp,
                                    uint32_t *d_text, uint32_t *d_suff, uint8_t *d_bwt, uint64_t *n_records, uint64_t *first_position);

/* Layout of the index files the shard was loaded from: byte widths of lcp (x), text (y), suff (z) and whether it
 * was the BCR triple.  Only the reference's post-EOF phantom record depends on it (DESIGN.md section 5).
 * e2s_shard_load_gesa sets (x, y, z, 0) itself; SoA loads default to (4, 4, 4, 0).  Call before e2s_shard_seal. */
int e2s_shard_set_layout(e2s_shard *sh, int x, int y, int z, int bcr);

/* Call once after the last load: on the last shard fills the records past n_global with the
 * reference's post-EOF phantom record (SURVEY.md §8(a) A3/B2; ref:clust2snp.cpp:827-833). */
int e2s_shard_seal(e2s_shard *sh);

/* Width in bytes of the LCP stream K1 reads for this shard: 1 when the seal found every LCP value <= 127 and
 * built the one-byte resident copy (what egsa's default 1-byte LCP files hold, ref:pipeline.sh:30-32), else 4.
 * Setting E2S_LCP_WIDE=1 in the environment before the seal keeps the 4-byte stream. */
int e2s_shard_lcp_bytes_resident(const e2s_shard *sh);

/* The index of the reads staged on the shard's context (e2s_reads_stage / _dev), built on the device straight into the
 * shard's own arrays: what e2s_shard_load_* of the X.gesa that `build_gesa -x x -y y -z z` writes would leave, without the
 * file (each field truncated to its width as that file holds it; the layout set as e2s_shard_set_layout(x, y, z, 0) does).
 * off = the staged collection's n_reads + 1 offsets in HOST memory (checked as the ragged builders check them).  The shard
 * must hold the whole eBWT: n_local = n_global = off[n_reads] + n_reads, global_off = 0, not chunked.  The whole index is
 * built in one call when its scratch fits 0.92 of the free device memory next to the shard and the reads, else key range by
 * key range (E2S_BUILD_RANGE_RECORDS forces ranges).  A base outside ACGT, a read of 65536 bases or more: E2S_ERR_UNSUPPORTED;
 * not even one key range fits: E2S_ERR_NOMEM.  Call e2s_shard_seal afterwards. */
int e2s_shard_build_egsa(e2s_shard *sh, const uint64_t *off, int x, int y, int z);

/* ---- one index over several shards, each built from the reads for its own key range -------------------------------------
 * Every shard (one per GPU, or several on one) stages all the reads, and
 *   1. e2s_reads_key_cuts      the same cuts on every shard (deterministic, no collective);
 *   2. e2s_shard_create        shard i: n_local = position[i+1] - position[i], global_off = position[i], n_global = position[parts];
 *   3. e2s_shard_build_egsa_range  shard i's key range [key_lo[i], key_lo[i+1]) (key_hi = 0 on the last shard);
 *   4. e2s_shard_halo_row      this shard's row, moved to every shard by the caller (host memory, torch.distributed, ...);
 *   5. e2s_shard_halo_apply    all rows in shard order, then e2s_shard_seal;
 * then the shards are what e2s_shard_load_* of the X.gesa of `build_gesa -x -y -z` with 2 positions of left and 151 of right halo
 * would leave, and the multi-shard sequence (e2s_cluster_run, e2s_exchange_finish / e2s_pipeline_sharded, ...) runs on them. */

/* Cuts of the key space (the builder's first key word: 32 symbols at 2 bits, A=0 C=1 G=2 T=3, first symbol most significant, zero
 * padded) into `parts` (1..1024) ranges of about equal size for the reads staged on ctx (off = their n_reads + 1 HOST offsets).
 * key_lo[0] = 0 < key_lo[1] < ... < key_lo[parts-1]; range i is [key_lo[i], key_lo[i+1]) (no upper bound for the last); position[i]
 * = the exact index position of cut i, position[parts] = off[n_reads] + n_reads.  Cuts are quantiles of the first key words of a
 * fixed-stride sample of the suffixes (no RNG: the same reads give the same cuts everywhere).  All suffixes of one key value stay in
 * one range, so a heavy value (e.g. the terminators, key 0) makes its range larger.  A range of fewer than 2 positions:
 * E2S_ERR_UNSUPPORTED (too many shards for this collection). */
int e2s_reads_key_cuts(e2s_ctx *ctx, const uint64_t *off, int parts, uint64_t *key_lo, uint64_t *position);
/* e2s_shard_build_egsa for the records of the key range [key_lo, key_hi) (key_hi = 0: no upper bound) only, written at the shard's
 * local positions: they must be its global positions [global_off, global_off + n_local) of an eBWT of n_global = off[n_reads] +
 * n_reads positions (E2S_ERR_ARG otherwise).  Resident shards only.  The range is built in one call when its scratch fits 0.92 of the
 * free device memory, else sub-range by sub-range.  lcp of the shard's position 0 is left at 0 when global_off > 0: the halo step
 * sets it.  e2s_shard_build_egsa is this call with key_lo = key_hi = 0 on a shard of the whole eBWT. */
int e2s_shard_build_egsa_range(e2s_shard *sh, const uint64_t *off, uint64_t key_lo, uint64_t key_hi, int x, int y, int z);
/* u64 words of one halo row: n_local, global_off, the ids (text << 32 | suff at full width) of the shard's first and last suffix,
 * then its last 2 and its first min(151, n_local) records as stored */
uint64_t e2s_shard_halo_row_words(void);
/* this built shard's halo row (row: e2s_shard_halo_row_words() words) */
int e2s_shard_halo_row(e2s_shard *sh, uint64_t *row);
/* rows = every shard's halo row in shard order (they must tile the eBWT; row `my` is this shard's).  Writes the left halo (the
 * previous shard's last 2 records), the right halo (the first records of the shards after this one, up to 151 or the end of the
 * eBWT) and this shard's lcp[0], every record that starts a shard carrying the LCP of the last suffix of the shard before it and its
 * own first suffix (the builder's rule on the staged reads, masked to the lcp width).  Call e2s_shard_seal afterwards. */
int e2s_shard_halo_apply(e2s_shard *sh, const uint64_t *rows, int n_shards, int my);

/* the read collection (FASTA bases), needed by e2s_find_events only: ref:clust2snp.cpp:147-212 */
int e2s_reads_stage(e2s_ctx *ctx, const uint8_t *bases, const uint64_t *offsets /* n_reads+1 */, uint64_t n_reads);
int e2s_reads_stage_dev(e2s_ctx *ctx, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n_reads,
                        uint64_t n_bases);

/* ---------------------------------------------------------------------------------------
 * phase 1: ebwt2clust  (cluster_lm + append_entry: ref:ebwt2clust.cpp:54-139)
 * ------------------------------------------------------------------------------------- */

/* What one shard knows after its scan; plain u64 words so it can be all-gathered as is. */
typedef struct {
    uint64_t n_local, global_off, n_global;
    uint64_t n_end;          /* closures (ENDs) inside the shard, head included */
    uint64_t n_written;      /* records with both ends known locally and length >= min_len */
    uint64_t head_end;       /* 1 + global position of an END whose START precedes the shard; 0 = none */
    uint64_t any_event;      /* shard contains at least one START or END */
    uint64_t open_start;     /* 1 + global START still open at the end of the shard; 0 = none */
    uint64_t end_nm2_start;  /* last shard: 1 + START of the cluster closed at n_global-2, 0 = none,
                                ~0 = that cluster is this shard's head (START unknown locally) */
    uint64_t tail_lcp_nm2, tail_lcp_nm1, tail_bwt_nm1; /* last shard: lcp[n-2], lcp[n-1], bwt[n-1] */
    uint64_t k, min_len;
    uint64_t lcp_bytes;      /* -x of the index files: the post-EOF phantom LCP is truncated to this width */
} e2s_cluster_summary;

/* Result of merging all shard summaries, from the point of view of shard `my`. */
typedef struct {
    uint64_t record_offset;  /* index in the global .clusters of this shard's first record */
    uint64_t total_written;  /* records in the global .clusters */
    uint64_t n_clust_out;    /* closures, as printed by ref:ebwt2clust.cpp:137 (low 32 bits are printed) */
    uint32_t phantom_lcp;    /* the post-EOF lcp value P that was applied */
    uint32_t n_prepend;      /* 0/1: this shard's head record (goes before its own records) */
    uint32_t n_append;       /* 0..2: tail records (last shard only; go after its own records) */
    uint32_t n_adopt;        /* 0..3: records written by a later shard (its head) or by the tail rule whose START
                                lies in this shard: phase 2 analyses them here */
    uint64_t prepend_start; uint64_t prepend_len; uint64_t prepend_written; /* written = passes min_len */
    uint64_t append_start[2]; uint64_t append_len[2];
    uint64_t adopt_start[3]; uint64_t adopt_len[3];
} e2s_cluster_merged;

/* Fused mode for callers that run both phases on resident data: from now on e2s_cluster_run also applies clust2snp's
 * BWT-only prefilter for this -m (find_variants, ref:clust2snp.cpp:402-429) while it writes the records, and a later
 * e2s_find_events with the same -m skips its own pass over the BWT.  0 switches it off (the default; the CLIs, which
 * are separate processes as in the reference, never use it).  Results are identical either way. */
int e2s_cluster_prefilter(e2s_shard *sh, int mcov_out);

/* K1+K2 on the shard: LCP boundary stencil + decoupled look-back scan + compaction.
 * Records stay on the device; *summary is written on the host. */
int e2s_cluster_run(e2s_shard *sh, uint32_t k, int32_t min_len, e2s_cluster_summary *summary);
/* Host-only integer logic (no CUDA): resolve shard heads, the tail + phantom rule, offsets. */
int e2s_cluster_merge(const e2s_cluster_summary *all, int n_shards, int my, e2s_cluster_merged *out);
/* Apply the merge to the device-resident record list of the shard (prepend/append records). */
int e2s_cluster_finalize(e2s_shard *sh, const e2s_cluster_merged *merged);
/* Single-shard convenience = run + merge(1 shard) + finalize; the whole of ebwt2clust's cluster_lm. */
int e2s_cluster_lm(e2s_shard *sh, uint32_t k, int32_t min_len, uint64_t *n_written, uint64_t *n_clust_out);

/* number of records in the shard's device list / copy them out (global start, wrapped u16 length) */
int e2s_cluster_count(const e2s_shard *sh, uint64_t *m);
int e2s_cluster_fetch(e2s_shard *sh, uint64_t *start, uint16_t *len, uint64_t cap, uint64_t *m);
/* same, as the 10-byte records of the .clusters file (ref:ebwt2clust.cpp:58-59) */
int e2s_cluster_fetch_packed(e2s_shard *sh, void *rec10, uint64_t cap_records, uint64_t *m);

/* ---------------------------------------------------------------------------------------
 * phase 2: clust2snp
 * ------------------------------------------------------------------------------------- */

/* Replace the shard's record list by records read from a .clusters file (clust2snp accepts the
 * output of any ebwt2clust run).  Records must be position-ordered and disjoint (what
 * ebwt2clust writes); anything else returns E2S_ERR_UNSUPPORTED. */
int e2s_clusters_stage_packed(e2s_shard *sh, const void *rec10, uint64_t m);
int e2s_clusters_stage(e2s_shard *sh, const uint64_t *start, const uint16_t *len, uint64_t m);

/* statistics(): ref:clust2snp.cpp:877-966.  The device part is the length histogram of the
 * shard's records; e2s_statistics_finish adds the reference's double count of the last record
 * and runs the pval loop (one IEEE double division per step, on the host as in the reference). */
typedef struct {
    uint64_t hist[E2S_HIST_BINS];
    uint64_t n_clust, n_bases;
    uint64_t last_len;  /* length of the shard's last record (valid if n_clust > 0) */
    uint64_t max_len;   /* filled by e2s_statistics_finish */
    int32_t max_clust_length;
    int32_t reserved;
} e2s_stats;
int e2s_statistics(e2s_shard *sh, e2s_stats *st);
int e2s_statistics_finish(e2s_stats *sum_over_shards, uint64_t last_len_global, int mcov_out, double pval);

/* Multi-shard glue between the phases, host-only: given the all-gathered scan summaries and the statistics of every
 * shard's OWN records (e2s_statistics before e2s_cluster_finalize), runs e2s_cluster_merge for all shards, adds the
 * records the merge creates at shard heads / at the tail and finishes statistics().  *mine = merged view of shard `my`. */
int e2s_exchange_finish(const e2s_cluster_summary *sums, const e2s_stats *own, int n_shards, int my, int mcov_out, double pval,
                        e2s_cluster_merged *mine, e2s_stats *total);

typedef struct {
    int32_t k_left;          /* -L 31 */
    int32_t k_right;         /* -R 30 */
    int32_t mcov_out;        /* -m 5  */
    int32_t max_gap;         /* -g 10 */
    int32_t consensus_reads; /* -c 20 */
    int32_t max_err;         /* -e 2  */
    int32_t max_snvs;        /* 3: ref:clust2snp.cpp:648 tests max_snvs_def, -v is dead */
    int32_t reserved;
    double pval;             /* -p 0.99 */
    uint64_t nr_reads1;      /* -n */
} e2s_snp_params;
void e2s_snp_default_params(e2s_snp_params *p);

/* one candidate that survived the support test (variant_t + distance(): ref:clust2snp.cpp:124-137,254-302) */
typedef struct {
    int32_t D;       /* mismatches outside the indel */
    int32_t gap;     /* 0 SNP, >0 insert in sample 0, <0 insert in sample 1 */
    int32_t supp0, supp1;
    int32_t right_len;
    int32_t keep;    /* 1 iff D <= max_snvs: the event is written to .snp */
    uint64_t cluster_start; /* provenance: global start of the cluster */
    char left0[E2S_MAX_K];
    char left1[E2S_MAX_K];
    char right[E2S_MAX_K];
} e2s_event;

typedef struct {
    uint64_t n_analysed;   /* clusters passing 2m <= len <= max_clust_length */
    uint64_t n_flagged;    /* of those, clusters passing find_variants' filters (ref:clust2snp.cpp:396-429) */
    uint64_t n_candidates; /* "Done. C potential variants detected" ref:clust2snp.cpp:859 */
    uint64_t n_variants;   /* supp0 > 0 and supp1 > 0, ref:clust2snp.cpp:595 */
    uint64_t n_events;     /* D <= 3, written to .snp */
    uint64_t saw_n;        /* an N/n met in BWT or contexts: the reference is non-deterministic there */
} e2s_snp_counts;

/* find_events(): K3 (per-cluster 2x4 histogram, first-argmax LCP, filters, ordered candidate
 * enumeration) + K4 (gSA-driven context gather, consensus, support, distance).
 * ref:clust2snp.cpp:367-500, 505-628, 254-302. */
int e2s_find_events(e2s_shard *sh, const e2s_snp_params *p, int max_clust_length, e2s_snp_counts *counts);
/* the n_variants surviving candidates in reference order */
int e2s_events_fetch(e2s_shard *sh, e2s_event *events, uint64_t cap, uint64_t *n);
/* to_file(): ref:clust2snp.cpp:633-780.  Host-only text formatting of the kept events; ids start
 * at first_id (1 for a single shard).  *text is malloc'ed: release with e2s_free. */
int e2s_events_format(const e2s_event *events, uint64_t n, uint64_t first_id, const e2s_snp_params *p,
                      char **text, size_t *len);
void e2s_free(void *p);

/* ---------------------------------------------------------------------------------------
 * chunked shards: inputs larger than device memory (BASELINE config 4).  The reference streams: ebwt2clust holds three
 * records at a time (ref:ebwt2clust.cpp:90-122), clust2snp one cluster and the candidates (ref:clust2snp.cpp:806-857).
 * Here a CHUNK IS A SHARD IN TIME: the device buffers of a chunked shard hold one chunk of the shard's range; chunks are
 * loaded and scanned one after the other with the open-cluster state carried over on the device side, each chunk's records
 * are handed out as soon as it is scanned, and the records of the clusters that survive the fused BWT prefilter are copied
 * to a compact payload, so that clust2snp's analysis runs once, after the last chunk, when statistics() has chosen
 * max_clust_length -- without a second pass over the index.  Resident footprint: 14.6 bytes x chunk_positions + the
 * payload (a few KB per candidate variant), whatever n is.
 *
 *   e2s_shard_create_chunked(ctx, n_local, global_off, n_global, chunk_positions, &sh);
 *   for every chunk [lo, lo + cn) of the range, in order (cn = e2s_shard_chunk_positions(sh), the last one may be shorter):
 *       e2s_chunk_begin(sh, lo, cn);
 *       e2s_shard_load_gesa / _soa / _soa_dev(...)   records [lo - 176, lo + cn + 152) as far as the eBWT reaches
 *       e2s_chunk_scan(sh, k, min_len, mcov_out, &m);  e2s_cluster_fetch_packed(sh, ...)  -> the chunk's m records
 *   e2s_chunked_finish(sh, k, min_len, &summary);  then, exactly as for a resident shard:
 *   e2s_cluster_merge -> e2s_cluster_finalize -> e2s_statistics (+ _finish) -> e2s_find_events -> e2s_events_fetch.
 * Needs the one-pass scan: every LCP value <= 127 (reads shorter than 128 bases) and -m <= 33 (else E2S_ERR_UNSUPPORTED).
 * ------------------------------------------------------------------------------------- */
int e2s_shard_create_chunked(e2s_ctx *ctx, uint64_t n_local, uint64_t global_off, uint64_t n_global, uint64_t chunk_positions,
                             e2s_shard **out);
uint64_t e2s_shard_chunk_positions(const e2s_shard *sh); /* positions per chunk (rounded up to whole scan tiles); 0: not chunked */
int e2s_chunk_begin(e2s_shard *sh, uint64_t chunk_lo, uint64_t chunk_n);
/* mcov_out = clust2snp's -m when both tools run (fused prefilter + capture), 0 for ebwt2clust alone */
int e2s_chunk_scan(e2s_shard *sh, uint32_t k, int32_t min_len, int mcov_out, uint64_t *n_records);
int e2s_chunked_finish(e2s_shard *sh, uint32_t k, int32_t min_len, e2s_cluster_summary *summary);
int e2s_chunked_reset(e2s_shard *sh); /* stream the range again from its first chunk */
/* clust2snp on a chunked shard (ref:clust2snp.cpp:788-872 streams the index past the .clusters records in the same way): after
 * the loads of a chunk, hand over the `m` records of the .clusters file whose START lies in the chunk (10 bytes each, file
 * order) instead of scanning for clusters; the BWT prefilter runs on them and the EGSA records of its survivors are kept.
 * max_clust_length = the result of statistics() over the whole file (e2s_statistics_finish).  After the last chunk
 * e2s_chunked_clusters_finish, then e2s_find_events / e2s_events_fetch as for any shard. */
int e2s_chunk_stage_clusters(e2s_shard *sh, const void *rec10, uint64_t m, int mcov_out, int max_clust_length,
                             uint64_t *n_survivors);
int e2s_chunked_clusters_finish(e2s_shard *sh);
/* Lean SoA inputs for a chunked shard: text / suff stay in the caller's pairSA buffer (suff(z) then text(y) per position, index =
 * global position; it must stay valid until the last e2s_chunk_scan), chunks are loaded with e2s_shard_load_lcp_bwt (lcp at x
 * bytes per position + BWT bytes: `lcp` / `bwt` point at the element of global position `first`), and e2s_chunk_scan fetches the
 * records of the clusters that survive the prefilter from the host.  pair_sa == NULL switches the mode off. */
int e2s_shard_host_gsa(e2s_shard *sh, const void *pair_sa, int y, int z);
int e2s_shard_load_lcp_bwt(e2s_shard *sh, const void *lcp, int x, const uint8_t *bwt, uint64_t first, uint64_t count);
/* The BCR triple as it is in the files (egsa_stream's second input format, ref:include.hpp:157-188): lcp at x bytes, BWT bytes,
 * pairSA = suff(z) then text(y) per position; every pointer at the element of global position `first`.  Split and widened on
 * the device.  Any shard; ebwt2clust needs e2s_shard_load_lcp_bwt only (the cluster scan never reads text / suff). */
int e2s_shard_load_bcr(e2s_shard *sh, const void *lcp, int x, const uint8_t *bwt, const void *pair_sa, int y, int z,
                       uint64_t first, uint64_t count);
/* Chunked shards on several GPUs (one process per GPU): after every rank's last chunk, e2s_chunked_finish + ONE ncclAllGather
 * of the ranks' accumulators + merge + statistics() + e2s_cluster_finalize.  Collective over the communicator. */
int e2s_chunked_exchange(e2s_shard *sh, e2s_comm *comm, uint32_t k, int32_t min_len, int mcov_out, double pval,
                         e2s_cluster_merged *merged, e2s_stats *stats);

/* ---------------------------------------------------------------------------------------
 * end-to-end convenience over host buffers (what bench.py's `e2e` times)
 * ------------------------------------------------------------------------------------- */
typedef struct {
    uint64_t n_written, n_clust_out;
    int32_t max_clust_length;
    int32_t reserved;
    e2s_snp_counts snp;
    uint64_t h2d_bytes, d2h_bytes;
} e2s_pipeline_result;

/* ebwt2clust + clust2snp on a sealed shard that holds the whole eBWT of one GPU, reads already staged:
 * cluster_lm + statistics + find_events (ref:ebwt2clust.cpp:194, ref:clust2snp.cpp:1080-1081) in one call.
 * Records and events stay on the shard (e2s_cluster_fetch*, e2s_events_fetch). */
int e2s_pipeline_resident(e2s_shard *sh, uint32_t k, int32_t min_len, const e2s_snp_params *p, e2s_pipeline_result *res);

/* One process per GPU (SURVEY.md 8(e)): the exchange between the phases inside the library.  A communicator wraps an
 * NCCL communicator created from a 128-byte unique id (made on one rank with e2s_comm_unique_id and handed to the others
 * by whatever launched the processes: torch.distributed in bench.py).  NCCL is bound at run time (libnccl.so.2).
 * e2s_pipeline_sharded = e2s_pipeline_resident for a shard of a sharded eBWT: the scan with clust2snp's BWT prefilter, ONE
 * ncclAllGather of every shard's scan accumulators on the context's stream, the merge and statistics() of all shards on the
 * device (identical on all ranks), K3x/K3b/K4 on the shard's survivors, one host synchronisation.  Needs valid clust2snp
 * parameters (E2S_ERR_UNSUPPORTED otherwise).  Collective: every rank of the communicator must call it. */
/* Host-only (no CUDA), exposed for tests and for callers that move the rows themselves: e2s_exchange_row_words() u64 words per
 * shard = the scan's device accumulators (ClusterDev: counters, open-cluster state, tail values, length histogram of the
 * shard's own records) followed by n_local, global_off, lcp_bytes, 0.  e2s_exchange_rows_finish turns the gathered rows
 * into summaries + own-record statistics and runs e2s_exchange_finish. */
uint64_t e2s_exchange_row_words(void);
int e2s_exchange_rows_finish(const uint64_t *rows, int n_shards, int my, uint64_t n_global, uint32_t k, int32_t min_len,
                             int mcov_out, double pval, e2s_cluster_merged *mine, e2s_stats *total);
int e2s_comm_unique_id(uint8_t *id128);
int e2s_comm_create(e2s_ctx *ctx, const uint8_t *id128, int rank, int world, e2s_comm **out);
/* A communicator whose all-gather the caller performs: where the library would call ncclAllGather it copies this rank's row
 * (`words` u64) to the host, synchronises the context's stream and calls fn(user, rank, world, send, recv, words).  fn must
 * return on every rank with recv = the `world` rows in rank order (the contract of ncclAllGather), and 0; any other value fails
 * the call with E2S_ERR_STATE.  The rows then go back to the device on the stream.  It lets several ranks of one sharded step
 * run in one process, on one GPU (threads and a barrier), so the multi-rank step is testable without several GPUs.  The
 * callback runs on the thread that made the library call. */
typedef int (*e2s_gather_fn)(void *user, int rank, int world, const uint64_t *send, uint64_t *recv, uint64_t words);
int e2s_comm_create_gather(e2s_ctx *ctx, int rank, int world, e2s_gather_fn fn, void *user, e2s_comm **out);
void e2s_comm_destroy(e2s_comm *comm);
int e2s_pipeline_sharded(e2s_shard *sh, e2s_comm *comm, uint32_t k, int32_t min_len, const e2s_snp_params *p,
                         e2s_cluster_merged *merged, e2s_stats *stats, e2s_snp_counts *counts);

/* ebwt2clust + clust2snp on one GPU from host buffers: .gesa records + reads in, .clusters
 * records (10-byte, into rec10 if non-NULL) and events out.  The records stream through a chunked shard of
 * E2S_CHUNK_POSITIONS positions (environment, default 2^28): device memory does not grow with n. */
int e2s_pipeline_host(e2s_ctx *ctx, const void *gesa_records, uint64_t n, int x, int y, int z,
                      const uint8_t *read_bases, const uint64_t *read_off, uint64_t n_reads,
                      uint32_t k, int32_t min_len, const e2s_snp_params *p,
                      void *rec10, uint64_t cap_records, e2s_event *events, uint64_t cap_events,
                      e2s_pipeline_result *res);

/* ebwt2clust + clust2snp from the reads alone, on one GPU: stage the reads (the only H2D), build the index into a resident
 * shard (e2s_shard_build_egsa), seal, e2s_pipeline_resident, then records / events out exactly as e2s_pipeline_host returns
 * them for the X.gesa of layout x/y/z.  res->h2d_bytes = reads + offsets.  The context's resident shard is kept for the next
 * call of the same n. */
int e2s_pipeline_reads(e2s_ctx *ctx, const uint8_t *read_bases, const uint64_t *read_off, uint64_t n_reads, int x, int y, int z,
                       uint32_t k, int32_t min_len, const e2s_snp_params *p, void *rec10, uint64_t cap_records,
                       e2s_event *events, uint64_t cap_events, e2s_pipeline_result *res);

/* The same from the BCR triple (ref:include.hpp:157-188: X.out.lcp = lcp(x) per position, X.out = BWT bytes, X.out.pairSA =
 * suff(z) then text(y) per position), LEAN: phase 1 and the BWT prefilter need the LCP and the BWT only, so 1 + x bytes per
 * position cross PCIe instead of the 13 of an EGSA record; the pairSA buffer stays on the host and only the records of the
 * clusters that reach phase 2 (~0.1 %) are fetched from it.  Same outputs as e2s_pipeline_host on the same index.  Needs the
 * one-pass scan (every LCP value <= 127, -m <= 33). */
int e2s_pipeline_host_soa(e2s_ctx *ctx, const void *lcp, int x, const uint8_t *bwt, const void *pair_sa, int y, int z, uint64_t n,
                          const uint8_t *read_bases, const uint64_t *read_off, uint64_t n_reads, uint32_t k, int32_t min_len,
                          const e2s_snp_params *p, void *rec10, uint64_t cap_records, e2s_event *events, uint64_t cap_events,
                          e2s_pipeline_result *res);

/* The same for ONE eBWT over the GPUs of a box, one process (rank) per GPU (SURVEY.md 8(e)): every rank streams its contiguous
 * range [range_lo, range_lo + range_n) of the records through a chunked shard -- it stages nothing but its range and the
 * halos -- then the ranks' summaries and own-record histograms are exchanged with one ncclAllGather, every rank merges,
 * finishes statistics() and runs phase 2 on the clusters it owns.  `records` points at the record of global position `first`
 * and must reach from max(0, range_lo - 176) to min(n_global, range_lo + range_n + 152).  rec10 (if non-NULL) receives this
 * rank's slice of the .clusters file: *n_records records that belong at index merged->record_offset.  Event ids are an
 * output-time matter: the caller numbers them from the ranks' n_events.  Collective: every rank of the communicator calls it. */
int e2s_pipeline_host_sharded(e2s_ctx *ctx, e2s_comm *comm, const void *records, uint64_t first, uint64_t range_lo,
                              uint64_t range_n, uint64_t n_global, int x, int y, int z, const uint8_t *read_bases,
                              const uint64_t *read_off, uint64_t n_reads, uint32_t k, int32_t min_len, const e2s_snp_params *p,
                              void *rec10, uint64_t cap_records, uint64_t *n_records, e2s_event *events, uint64_t cap_events,
                              e2s_cluster_merged *merged, e2s_stats *stats, e2s_pipeline_result *res);

#ifdef __cplusplus
}
#endif
#endif /* EBWT2SNP_B200_H */
