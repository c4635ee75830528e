// Internal declarations shared by the .cu translation units (not part of the C ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ebwt2snp_b200.h"

#include <vector>

namespace e2s {

// CUDA-event timing of selected kernels on the launch stream (enabled by e2s_ctx_timing)
struct KernelTimer {
    bool enabled = false;
    struct Rec { int id; cudaEvent_t a, b; };
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;  // events are reused: creating one costs microseconds on the launching thread
    cudaEvent_t take() {
        cudaEvent_t e;
        if (!pool.empty()) {
            e = pool.back();
            pool.pop_back();
        } else {
            cudaEventCreate(&e);
        }
        return e;
    }
    void give(cudaEvent_t e) { pool.push_back(e); }
    void begin(int id, cudaStream_t s) {
        if (!enabled) return;
        Rec r;
        r.id = id;
        r.a = take();
        r.b = take();
        cudaEventRecord(r.a, s);
        recs.push_back(r);
    }
    void end(cudaStream_t s) {
        if (!enabled || recs.empty()) return;
        cudaEventRecord(recs.back().b, s);
    }
};

// ---- phase 1 ---------------------------------------------------------------------------------
// One cluster handed to the exact test of phase 2 (find_variants, ref:clust2snp.cpp:367-500).  `base` is the index of the
// cluster's first record in the arrays phase 2 reads: the shard's resident arrays (start - global_off) or, in streaming
// mode, the compact payload the chunk's records were copied to before the chunk left the device.
struct SurvEntry {
    uint64_t start;  // global START (provenance; the events are put into eBWT order by it)
    uint64_t base;
    uint32_t len;    // wrapped 16-bit length, as in the .clusters record
    uint32_t pad;
};

struct ClusterDev {  // device-resident accumulators of one e2s_cluster_run (zeroed before the launch)
    unsigned long long n_end;
    unsigned long long n_written;
    unsigned long long head_end;       // 1 + global END position, 0 = none
    unsigned long long any_event;
    unsigned long long open_start;     // 1 + global START, 0 = none
    unsigned long long end_nm2_start;  // 1 + START of the cluster closed at n_global-2; ~0 = head; 0 = none
    unsigned long long overflow;
    unsigned long long ticket;         // K2's chunk dispenser
    unsigned long long n_pf;           // fused prefilter: clusters appended to (or dropped from, beyond its capacity) the survivor list
    unsigned long long last_rec;       // (index of the last kept record + 1) << 16 | its length
    unsigned long long tail_lcp_nm2, tail_lcp_nm1, tail_bwt_nm1;  // last shard: lcp[n-2], lcp[n-1], bwt[n-1]
    unsigned long long n_bases;        // sum of the kept records' lengths
    unsigned long long hist[E2S_HIST_BINS];  // their length histogram (lengths <= 150)
};

// ---- the exchange between the phases (merge.cu) -------------------------------------------------------
// one exchange row per shard: the scan's device accumulators + what the other ranks cannot know
constexpr size_t XR_DEV_WORDS = sizeof(ClusterDev) / 8;
constexpr size_t XR_WORDS = XR_DEV_WORDS + 4;  // + n_local, global_off, lcp_bytes, reserved
constexpr int MERGE_MAX_SHARDS = 64;
struct MergeOut {  // written by k_merge_stats
    e2s_cluster_merged mine;  // this shard's view of the merge
    e2s_stats total;          // statistics() over all shards' records, max_clust_length included
    int32_t status;           // merge.cuh: MERGE_OK ...
    int32_t pad;
};
struct MergeParams {
    const unsigned long long* rows;  // `world` rows of XR_WORDS words, in shard order (device memory)
    int world, my;
    uint64_t n_global;
    uint32_t k;
    int32_t min_len;
    int32_t mcov;
    double pval;
    uint64_t own_global_off;
    MergeOut* out;
    SurvEntry* pf_list;              // the records this shard adopts are appended here (null: no fused prefilter)
    uint64_t pf_cap;
    ClusterDev* res;                 // ... and counted in res->n_pf
};
cudaError_t launch_pack_exchange(const ClusterDev* res, uint64_t n_local, uint64_t global_off, uint64_t lcp_bytes, uint64_t* row,
                                 cudaStream_t stream);
cudaError_t launch_merge_stats(const MergeParams& p, cudaStream_t stream);

struct FlagParams {  // K1
    const uint32_t* lcp;  // local position 0 (PAD_L readable elements before it)
    uint64_t n_local, global_off, n_global;
    uint32_t k;
    uint32_t num_tiles;  // filled by the launcher
    uint32_t* s_words;   // START bit mask, bit i of word w = local position 32 w + i
    uint32_t* e_words;   // END bit mask
};

struct EmitParams {  // K2
    const uint32_t* s_words;
    const uint32_t* e_words;
    uint64_t num_tiles;
    uint64_t global_off, n_global;
    int32_t min_len;
    uint64_t* out_start;
    uint16_t* out_len;
    uint64_t cap;
    uint64_t* desc;      // chunk descriptors (emit_desc_words() words, zeroed before the launch)
    // fused BWT prefilter of find_variants (pipeline mode: the caller already knows clust2snp's -m); pf_mcov = 0: off
    const uint4* planes;            // the shard's resident base-code bit planes (planes.cuh)
    uint32_t pf_mcov;
    SurvEntry* pf_list;             // out: clusters that need the exact test, unordered
    uint64_t pf_cap;
    ClusterDev* res;
    const uint32_t* tail_lcp;  // &lcp[n_global-2] when this is the last shard, else null
    const uint8_t* tail_bwt;   // &bwt[n_global-1]
};

// k_cluster_scan (scan.cu): K1 + K2 in one pass over the bit-sliced LCP, one CTA per chunk of consecutive tiles
constexpr uint32_t SCAN_MAX_CHUNKS = 1024;
constexpr int LCPT_BLOCK = 2048;  // positions (= bytes) per block of the bit-sliced LCP; one block of padding before local position 0
inline size_t lcpt_bytes(uint64_t alloc_r) { return size_t(alloc_r) + 2 * LCPT_BLOCK; }  // ... and one after the last tile
struct ChunkRec {  // what a chunk leaves behind (zeroed before the launch)
    unsigned long long own_count;   // records in the chunk's segment (all ENDs with a START inside the chunk, minus the short ones)
    unsigned long long head_end;    // 1 + global position of the chunk's first event if that is an END, 0 = none
    unsigned long long last_state;  // 0: no event in the chunk; 1: closed after it; >= 2: 2 + global START left open
    unsigned long long n_end;       // ENDs in the chunk, head included
    unsigned long long n_bases;     // sum of the lengths in the segment
    unsigned long long last_len;    // length of the segment's last record
    unsigned long long pad[2];
};
struct ChunkSeg {  // written by k_chunk_resolve: where the chunk's records go in the position-ordered list
    unsigned long long off;         // index of the chunk's first record (its head record if kept, else its segment's first)
    unsigned long long own_count;
    unsigned long long head_start;
    uint32_t head_len, head_kept;
};
struct Scan8Params {
    const uint8_t* lcpt;        // the bit-sliced LCP (k_derive): blocks of LCPT_BLOCK positions = 8 runs (planes 0..6, A) of 32 words;
                                // byte 0 = block of the local positions -LCPT_BLOCK .. -1, lcpt_bytes(alloc_r) bytes in all
    const uint4* planes;        // resident base-code bit planes (fused prefilter)
    uint64_t n_local, global_off, n_global;
    uint32_t k;
    int32_t min_len;            // <= 33
    uint32_t num_tiles;         // filled by the launcher
    uint32_t km[8];             // (launcher) bit b of min(k, 128) as an all-ones / zero word, b < 7; [7]: k >= 128
    uint32_t t_int_lo, t_int_hi;  // (launcher) tiles that need none of the edge rules
    uint32_t n_chunks, tiles_per_chunk;  // scan_plan
    uint64_t* seg_start;        // record segments: chunk c owns [c * seg_cap, (c + 1) * seg_cap)
    uint16_t* seg_len;
    uint64_t seg_cap;
    ChunkRec* chunks;
    uint32_t pf_mcov;
    SurvEntry* pf_list;
    uint64_t pf_cap;
    ClusterDev* res;
    const uint32_t* tail_lcp;   // &lcp[n_global-2] when this is the last shard, else null
    const uint8_t* tail_bwt;    // &bwt[n_global-1]
};
struct ResolveParams {  // k_chunk_resolve
    const ChunkRec* chunks;
    ChunkSeg* segs;
    uint32_t n_chunks;
    int32_t min_len;
    uint64_t global_off, n_global;
    uint64_t init_state;        // open-cluster state before the shard: 0 closed (eBWT start), 1 unknown (an earlier shard decides)
    const uint4* planes;
    uint32_t pf_mcov;
    SurvEntry* pf_list;
    uint64_t pf_cap;
    ClusterDev* res;
};
uint64_t scan_num_tiles(uint64_t n_local);
cudaError_t scan_plan(uint64_t n_local, int sm_count, uint32_t* n_chunks, uint32_t* tiles_per_chunk);
cudaError_t launch_scan(const Scan8Params& p, uint64_t alloc_r, cudaStream_t stream);
cudaError_t launch_chunk_resolve(const ResolveParams& p, cudaStream_t stream);
// segments -> contiguous: SoA (out_start / out_len) or 10-byte file records (out_packed); the other output(s) null
cudaError_t launch_export_records(const ChunkSeg* segs, uint32_t n_chunks, uint64_t seg_cap, const uint64_t* seg_start,
                                  const uint16_t* seg_len, uint64_t* out_start, uint16_t* out_len, uint8_t* out_packed,
                                  cudaStream_t stream);

uint64_t flags_words_needed(uint64_t n_local);
uint64_t emit_num_tiles(uint64_t n_local);
uint64_t emit_desc_words();
cudaError_t launch_flags(const FlagParams& p, uint64_t rows_alloc32, int sm_count, cudaStream_t stream);
cudaError_t launch_emit(const EmitParams& p, int sm_count, cudaStream_t stream);
// small helpers: append up to 3 records to the device list / pack the list into 10-byte file records
cudaError_t launch_put_records(uint64_t* d_start, uint16_t* d_len, uint64_t at, const uint64_t* st, const uint64_t* ln,
                               int n, cudaStream_t stream);
cudaError_t launch_pack_records(const uint64_t* d_start, const uint16_t* d_len, uint64_t m, uint8_t* d_out,
                                cudaStream_t stream, int sm_count);

// ---- staging -----------------------------------------------------------------------------------
// AoS records -> SoA.  d_rec: `count` records of (y+z+x+1) bytes; outputs are pointers to the element
// that receives record 0 (any may be null).
cudaError_t launch_unpack_gesa(const uint8_t* d_rec, uint64_t count, int x, int y, int z, uint32_t* lcp, uint32_t* text,
                               uint32_t* suff, uint8_t* bwt, cudaStream_t stream, int sm_count);
// narrow resident copies of the local positions [a, b) just loaded (byte LCP + base-code bit planes); *flag |= 1 when an
// LCP value in [chk_lo, chk_hi) does not fit the byte copy
cudaError_t launch_derive(const uint32_t* lcp, const uint8_t* bwt, uint8_t* lcpt, uint4* planes, int64_t a, int64_t b,
                          int64_t chk_lo, int64_t chk_hi, uint32_t* flag, cudaStream_t stream, int sm_count);
cudaError_t launch_widen(const uint8_t* d_src, int w, uint32_t* d_dst, uint64_t cnt, cudaStream_t stream, int sm_count);
cudaError_t launch_widen_pairs(const uint8_t* d_src, int wa, int wb, uint32_t* d_a, uint32_t* d_b, uint64_t cnt, cudaStream_t stream,
                               int sm_count);
cudaError_t launch_fill_phantom(uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt, uint64_t n_local,
                                uint64_t count, int x, int y, int z, int bcr, cudaStream_t stream);

// ---- EGSA construction (build_egsa.cu) -----------------------------------------------------------
// What the builder keeps of each output value: the field widths of a .gesa file (lcp mod 2^(8x), text mod 2^(8y), suff mod 2^(8z),
// as its writer truncates them); all ones = the full values
struct FieldMask {
    uint32_t lcp = ~0u, text = ~0u, suff = ~0u;
};

// suffix sort of R reads (device pointer, no separators) -> lcp/text/suff/bwt device arrays of total_bases + R elements; synchronises.
// d_off == nullptr: every read has L bases; else R + 1 DEVICE offsets (h_off: the same in host memory) and L = the longest read (< 65536).
// cudaErrorInvalidValue = a base outside ACGT / acgt; cudaErrorInvalidConfiguration = a read of 65536 bases or more.
cudaError_t build_egsa(const uint8_t* d_reads, const uint64_t* d_off, const uint64_t* h_off, uint64_t R, uint32_t L, uint64_t total_bases,
                       uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, cudaStream_t stream, uint64_t* launches,
                       FieldMask mask = FieldMask(), uint64_t* ends = nullptr);

// one key range of the index (see build_egsa.cu); reads as for build_egsa (d_off == nullptr: R reads of L bases), no host offsets needed;
// cudaErrorInvalidPitchValue = more than `cap` records (*n_out says how many).  ends (of both builders; when not null, and the range is
// not empty) = the first and the last record written as text << 32 | suff at full width, whatever the mask: the `before` of the next
// range, and the ends a shard's halo row carries
cudaError_t build_egsa_range(const uint8_t* d_reads, const uint64_t* d_off, uint64_t R, uint32_t L, uint64_t total_bases, uint64_t key_lo,
                             uint64_t key_hi, uint64_t before, uint64_t cap, uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt,
                             uint64_t* n_out, uint64_t* first_out, cudaStream_t stream, uint64_t* launches, FieldMask mask = FieldMask(),
                             uint64_t* ends = nullptr);

// Cuts of the key space into `parts` ranges of about equal size (see build_egsa.cu): key_lo[0] = 0 < key_lo[1] < ... (the first key
// words, as for build_egsa_range), position[i] = the index position of cut i, position[parts] = total_bases + R.  Deterministic: a
// fixed-stride sample of the suffix slots, no RNG.  Reads as for build_egsa_range.  cudaErrorInvalidValue = a base outside ACGT / acgt.
cudaError_t key_cuts(const uint8_t* d_reads, const uint64_t* d_off, uint64_t R, uint32_t L, uint64_t total_bases, uint32_t parts,
                     uint64_t* key_lo, uint64_t* position, cudaStream_t stream, uint64_t* launches);

// lcp[j] = the builder's LCP (capped at the shorter suffix, never across a terminator) of the suffixes pairs[2 j] and pairs[2 j + 1]
// (text << 32 | suff, device memory) of the reads `bases` / R + 1 DEVICE offsets `off`, masked with lcp_mask; one launch, no sync
cudaError_t launch_pair_lcp(const uint8_t* bases, const uint64_t* off, const uint64_t* pairs, uint32_t n_pairs, uint32_t lcp_mask,
                            uint32_t* lcp, cudaStream_t stream);

// ---- phase 2 -----------------------------------------------------------------------------------
struct SnpDev {  // device counters of one e2s_find_events
    unsigned long long n_analysed;
    unsigned long long n_survivors;  // clusters that pass the base-code prefilter
    unsigned long long n_flagged;
    unsigned long long n_slots_valid;
    unsigned long long saw_n;
    unsigned long long bad_ref;
    unsigned long long unsorted;
    unsigned long long n_variants;   // candidates with supp0 > 0 and supp1 > 0
    unsigned long long n_events;     // of those, D <= max_snvs
    unsigned long long compact;      // K4 wrote the compact event records (reads hold nothing but upper-case ACGT, k_left / k_right <= 32)
};

struct SnpArrays {
    const uint32_t* lcp;
    const uint32_t* text;
    const uint32_t* suff;
    const uint8_t* bwt;   // all: local position 0
    const uint4* planes;  // resident base-code bit planes (planes.cuh), built at seal
    uint64_t n_local, global_off;
    const uint64_t* cl_start;  // global starts, sorted
    const uint16_t* cl_len;
    uint64_t m;
    const uint32_t* reads_flag = nullptr;  // two device words written when the reads were staged (launch_reads_check); null: unknown
};

struct CandSlot {  // one (flagged cluster, allele pair) slot written by K3b
    uint32_t n0, n1;
    uint32_t valid;
    uint32_t pad;
    uint64_t right_idx, right_pos;
    uint64_t cluster_start;
    // followed in the slot arrays by idx/pos lists (see snp.cu)
};

cudaError_t launch_len_hist(const uint16_t* len, uint64_t m, unsigned long long* hist /*151 + n_bases*/,
                            cudaStream_t stream, int sm_count);
cudaError_t launch_check_sorted(const uint64_t* start, const uint16_t* len, uint64_t m, SnpDev* dev,
                                cudaStream_t stream, int sm_count);

// Streaming (a shard processed chunk by chunk): before a chunk leaves the device, the records of its surviving clusters
// are copied to a compact payload (same four arrays, `base` of the entry = offset in them), so that phase 2 can run after
// the last chunk -- when max_clust_length is known -- without a second pass over the input.
struct CaptureParams {
    const SurvEntry* in;               // the chunk's survivors (base = index relative to the chunk's local position 0, may be negative)
    const unsigned long long* n_in;    // device-resident count (capped at n_in_cap)
    uint64_t n_in_cap;
    const uint32_t* lcp;
    const uint32_t* text;
    const uint32_t* suff;
    const uint8_t* bwt;                // the chunk's arrays, local position 0
    uint32_t* p_lcp;
    uint32_t* p_text;
    uint32_t* p_suff;
    uint8_t* p_bwt;                    // payload arrays
    uint64_t pay_cap;
    SurvEntry* out;                    // the shard's survivor list (entries with payload offsets)
    uint64_t out_cap;
    unsigned long long* counters;      // [0] payload cursor, [1] entries in `out`, [2] error bits: 1 = cluster not resident, 2 = payload full, 4 = list full
};
cudaError_t launch_capture(const CaptureParams& p, cudaStream_t stream, int sm_count);
cudaError_t launch_code_scan(const SnpArrays& a, uint32_t mcov, uint32_t max_len, SurvEntry* out, uint64_t cap, SnpDev* dev,
                             cudaStream_t stream, int sm_count);

// *flag |= 1 when one of the n bytes is not in ACGTacgt (K4 then keeps base_to_int's "anything else counts as A" path)
// flag[1] |= 1 unless all n_reads reads (offsets d_off[0 .. n_reads]) have the same length
cudaError_t launch_reads_check(const uint8_t* d_bases, uint64_t n, const uint64_t* d_off, uint64_t n_reads, uint32_t* flag, cudaStream_t stream,
                               int sm_count);

struct SnpWork;  // opaque scratch owned by the shard (snp.cu)
SnpWork* snp_work_create();
void snp_work_destroy(SnpWork* w);
// Runs K3a/K3x/K3b/K4 back to back on the stream with device-resident counts and synchronises ONCE at the
// end; the packed events are written by K4 straight into pinned host memory.  If a capacity guess
// (survivor / flagged lists) was too small the pass is repeated with larger buffers.
// pre_list: survivors of the prefilter when the scan already ran it (fused mode), else null.  Their number is pre_count, or
// -- d_pre_count != null -- a device-resident count (capped at pre_count = the list's capacity).  d_max_len != null: the
// exact test reads max_clust_length from device memory (written by the merge kernel earlier on the stream).
cudaError_t snp_run(SnpWork* w, const SnpArrays& a, const e2s_snp_params& p, int max_clust_length,
                    const uint8_t* d_read_bases, const uint64_t* d_read_off, uint64_t n_reads, int sm_count,
                    cudaStream_t stream, e2s_snp_counts* counts, uint64_t* launches, const char** err,
                    KernelTimer* timer, const SurvEntry* pre_list, uint64_t pre_count,
                    const unsigned long long* d_pre_count = nullptr, const int32_t* d_max_len = nullptr, bool sync = true);
// the counters of the last snp_run (valid after the stream has been synchronised); false: a capacity guess was too small
bool snp_collect(SnpWork* w, e2s_snp_counts* counts, const char** err, cudaError_t* rc);
cudaError_t snp_fetch_events(SnpWork* w, e2s_event* host, uint64_t cap, uint64_t* n, cudaStream_t stream);
uint32_t snp_event_stride(const SnpWork* w);  // bytes per candidate K4 wrote to pinned host memory in the last pass

}  // namespace e2s
