// EGSA construction on the GPU (SURVEY.md §8(f) rank 1): eBWT + LCP + generalized suffix array of a collection of
// reads, the input the two tools expect an external `egsa` / BCR run to have produced (ref:README.md:46-60,
// ref:pipeline.sh:98-109).  Reads may have any lengths (the reference accepts any FASTA, ref:clust2snp.cpp:147-212).
// Conventions = the ones this repo's synthetic data has used from the start (ebwt2snp_b200/synth.py; the reference pins
// none of them, SURVEY.md §8(b) last row):
//   one record per suffix of every read INCLUDING the terminator suffix (n = sum of (len_r + 1));
//   `$` < A < C < G < T; equal suffixes ordered by read id;
//   lcp[i] = common prefix with record i - 1, never extending over a terminator, lcp[0] = 0;
//   text = read id, suff = offset of the suffix in its read (len_r for the terminator suffix);
//   bwt = preceding character, `$` for whole-read suffixes.
//
// Suffixes of short reads are short strings, so there is no doubling: every suffix is a fixed-width key and the sort is
// a least-significant-digit radix sort written for exactly this key shape -- no library sort.
//   k_pack_reads   2 bits per base (A=0 C=1 G=2 T=3, most significant first), zero padded; read r's row starts at word
//                  (start_r >> 5) + 2 r (rows cannot overlap, no prefix sum over the reads needed)
//   k_init_ids     the initial order.  Equal lengths: id = (L - p) R + r, ascending = shortest suffix first, then read id.
//                  Ragged: id = (r << shift) | p in (read, offset) order, then one or two radix passes on the suffix
//                  LENGTH bring it to the same shortest-first order.
//   per key word w, last word first (zero padding orders a suffix before every longer one it prefixes because the sort is
//   stable and starts shortest-first).  A digit place moves only the suffixes long enough to have a symbol in it: the
//   others have digit 0 there, are still a prefix of the shortest-first order and stay where they are (L = 100: 13 passes'
//   worth of pairs instead of 25):
//     k_keys_hist  symbols [p + 32 w, p + 32 w + 32) of every suffix as one 64-bit word (funnel shift of two packed
//                  words) in the current id order, AND the 256-bin histograms of every 8-bit digit of that word in the
//                  same pass (shared-memory atomics; digit 0, which the zero padding makes the common one, by one ballot and
//                  one atomic per warp)
//     k_scan_hist  exclusive scans -> first output slot of every (digit place, bin)
//     k_radix_pass one launch per digit place that can differ (only the bits of symbols that exist in the longest read):
//                  tiles of 4096 pairs dealt by a ticket, stable warp-level multisplit (match.any), chained-scan
//                  decoupled look-back per bin, four tiles at a time (one 64-bit tagged word per tile and bin: no clearing
//                  between passes), keys and ids staged together in shared memory in output order and written in one sweep,
//                  so every bin leaves as a coalesced run.  The last place of a word moves the ids only.
//   key ranges     k_range_select / k_scan_chunks pick the suffixes whose first key word lies in [lo, hi) -- a contiguous range
//                  of the index -- and the same sort runs on those alone (build_egsa_range).  Equal lengths: the selected ids are
//                  already shortest first.  Ragged: they come in (read, offset) order and the length pass sorts them as above.
//   k_egsa_finish  decode (r, p); text, suff, bwt; lcp with the previous record = min(len_a - p_a, len_b - p_b, first
//                  differing symbol) by clz on XORed key words.
// Ids are 32-bit when they fit (equal lengths: n < 2^32; ragged: R << shift <= 2^32), else 64-bit.
// Outputs go straight to device arrays (a shard's resident SoA arrays via e2s_shard_load_soa_dev, or the caller's).

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <vector>

#include "common.cuh"
#include "internal.h"

namespace e2s {

namespace {

constexpr uint32_t LEN_WORD = 0xffffffffu;  // k_keys_hist: key = suffix length instead of a symbol word

struct ReadsView {
    const uint8_t* bases;  // all reads, no separators
    const uint64_t* off;   // R + 1 offsets into bases, or nullptr: equal lengths (read r starts at r * L)
    uint64_t R;
    uint32_t L;      // the read length (equal) / the longest read (ragged)
    uint32_t shift;  // ragged ids: (r << shift) | p; 0 = equal-length ids (L - p) R + r
    __device__ __forceinline__ uint64_t start(uint64_t r) const { return off ? off[r] : r * L; }
    __device__ __forceinline__ uint32_t len(uint64_t r) const { return off ? uint32_t(off[r + 1] - off[r]) : L; }
    __device__ __forceinline__ uint64_t row(uint64_t r, uint64_t st) const { return (st >> 5) + 2 * r; }
    template <typename IdT>
    __device__ __forceinline__ void decode(IdT id, uint64_t& r, uint32_t& p) const {
        if (shift) {
            r = uint64_t(id) >> shift;
            p = uint32_t(id) & ((1u << shift) - 1u);
        } else if (sizeof(IdT) == 4) {
            const uint32_t q = uint32_t(id) / uint32_t(R);
            r = uint32_t(id) - q * uint32_t(R);
            p = L - q;
        } else {
            const uint64_t q = uint64_t(id) / R;
            r = uint64_t(id) - q * R;
            p = L - uint32_t(q);
        }
    }
};

__device__ __forceinline__ uint32_t code2(uint32_t c) {  // ACGT / acgt -> 0..3 (anything else is refused by k_pack_reads)
    const uint32_t u = c & 0xDFu;
    return uint32_t(u == 'C') + 2u * uint32_t(u == 'G') + 3u * uint32_t(u == 'T');
}

// bits of x spread to the even positions of a 64-bit word
__device__ __forceinline__ uint64_t spread_even(uint32_t x) {
    uint64_t v = x;
    v = (v | (v << 16)) & 0x0000ffff0000ffffull;
    v = (v | (v << 8)) & 0x00ff00ff00ff00ffull;
    v = (v | (v << 4)) & 0x0f0f0f0f0f0f0f0full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v;
}

// one warp per read; per row word the lanes load 32 consecutive bases, two ballots collect the code bits, lane 0's symbol ends
// up in the two most significant bits.  The row has ceil(len / 32) + 1 words, the last one all padding.
// *bad is raised when a base is not one of ACGT / acgt: the 2-bit keys have no code for it (N would sort and compare as A)
__global__ void k_pack_reads(ReadsView v, uint64_t* __restrict__ packed, uint32_t* __restrict__ bad) {
    const uint64_t r = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (r >= v.R) return;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t st = v.start(r);
    const uint32_t len = v.len(r), W = (len + 31) >> 5;
    uint64_t* row = packed + v.row(r, st);
    bool other = false;
    for (uint32_t w = 0; w <= W; ++w) {
        const uint32_t s = 32 * w + lane;
        uint32_t code = 0;
        if (s < len) {
            const uint32_t c = v.bases[st + s], u = c & 0xDFu;
            other |= !(u == 'A' || u == 'C' || u == 'G' || u == 'T');
            code = code2(c);
        }
        const uint32_t lo = __brev(__ballot_sync(0xffffffffu, code & 1u)), hi = __brev(__ballot_sync(0xffffffffu, code & 2u));
        if (lane == 0) row[w] = (spread_even(hi) << 1) | spread_even(lo);
    }
    if (other) *bad = 1u;
}

// symbols [p + 32 w, +32) of a read as one word (zero past its end); row = the read's first packed word
__device__ __forceinline__ uint64_t suffix_word(const uint64_t* __restrict__ row, uint32_t len, uint32_t p, uint32_t w) {
    const uint32_t s = p + 32 * w;
    if (s >= len) return 0;
    const uint32_t q = s >> 5, sh = (s & 31) * 2;  // q < ceil(len / 32): row[q + 1] exists
    const uint64_t a = row[q];
    return sh ? (a << sh) | (row[q + 1] >> (64 - sh)) : a;
}

template <typename IdT>
__global__ void k_init_ids_equal(IdT* __restrict__ ids, uint64_t n) {
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) ids[i] = IdT(i);
}

// ragged: one warp per read; suffix (r, p) sits at start_r + r + p in the initial order
template <typename IdT>
__global__ void k_init_ids_ragged(ReadsView v, IdT* __restrict__ ids) {
    const uint64_t r = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (r >= v.R) return;
    const uint64_t st = v.start(r);
    const uint32_t len = v.len(r);
    for (uint32_t p = threadIdx.x & 31; p <= len; p += 32) ids[st + r + p] = IdT((r << v.shift) | p);
}

// ---- the radix sort ------------------------------------------------------------------------------------------------------
constexpr int RS_TILE = 4096;                   // pairs per tile (256 threads x 16 or 512 threads x 8)
constexpr int MAX_PLACES = 8;                   // 8-bit digit places in a 64-bit word

// tile status word of the chained scan: [63:45] tag of the pass (never 0), [44] inclusive, [43:0] count
constexpr int TAG_SHIFT = 45;
constexpr uint64_t INCL_BIT = uint64_t(1) << 44;
constexpr uint64_t CNT_MASK = INCL_BIT - 1;

__device__ __forceinline__ void st_status(uint64_t* d, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(d), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_status(const uint64_t* d) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(d) : "memory");
    return v;
}

// keys of word w in the current id order + the histograms of its `places` digit places (place j = bits [begin_bit + 8 j, +8))
template <typename IdT>
__global__ void __launch_bounds__(256) k_keys_hist(ReadsView v, const uint64_t* __restrict__ packed, const IdT* __restrict__ ids,
                                                   uint64_t n, uint32_t w, uint32_t begin_bit, uint32_t places,
                                                   uint64_t* __restrict__ keys, uint64_t* __restrict__ keys_alt, uint64_t dup,
                                                   unsigned long long* __restrict__ hist) {
    __shared__ uint32_t s_hist[MAX_PLACES][256];
    for (uint32_t b = threadIdx.x; b < MAX_PLACES * 256; b += blockDim.x) (&s_hist[0][0])[b] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    for (uint64_t base = uint64_t(blockIdx.x) * blockDim.x; base < n; base += uint64_t(gridDim.x) * blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        const bool valid = i < n;
        uint64_t key = 0;
        if (valid) {
            uint64_t r;
            uint32_t p;
            v.decode(ids[i], r, p);
            const uint64_t st = v.start(r);
            const uint32_t len = v.len(r);
            key = w == LEN_WORD ? uint64_t(len - p) : suffix_word(packed + v.row(r, st), len, p, w);
            keys[i] = key;
            if (i < dup) keys_alt[i] = key;  // not moved by the first places: wanted in whichever buffer is current later
        }
        for (uint32_t j = 0; j < places; ++j) {
            // zero padding makes digit 0 the common one in the low places: one atomic per warp for it, plain ones for the rest
            const uint32_t d = uint32_t(key >> (begin_bit + 8 * j)) & 0xffu;
            const uint32_t z = __ballot_sync(0xffffffffu, valid && d == 0);
            if (lane == 0 && z) atomicAdd(&s_hist[j][0], uint32_t(__popc(z)));
            if (valid && d) atomicAdd(&s_hist[j][d], 1u);
        }
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < places * 256; b += blockDim.x) {
        const uint32_t c = (&s_hist[0][0])[b];
        if (c) atomicAdd(hist + b, static_cast<unsigned long long>(c));
    }
}

struct PlaceSkip {
    uint64_t n[MAX_PLACES];  // leading suffixes of the word's range that place j leaves alone (all of them have digit 0 there)
};

// hist[place][bin] -> first output slot of the bin among the suffixes the place sorts (exclusive scan per place); clears hist
__global__ void k_scan_hist(unsigned long long* __restrict__ hist, uint64_t* __restrict__ bin_base, PlaceSkip skip) {
    __shared__ uint64_t s[MAX_PLACES][256];
    for (uint32_t b = threadIdx.x; b < MAX_PLACES * 256; b += blockDim.x) {
        (&s[0][0])[b] = hist[b];
        hist[b] = 0;
    }
    __syncthreads();
    if (threadIdx.x < MAX_PLACES) {
        uint64_t sum = 0;
        for (int b = 0; b < 256; ++b) {
            uint64_t t = s[threadIdx.x][b];
            if (b == 0) t = t > skip.n[threadIdx.x] ? t - skip.n[threadIdx.x] : 0;
            s[threadIdx.x][b] = sum;
            sum += t;
        }
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < MAX_PLACES * 256; b += blockDim.x) bin_base[b] = (&s[0][0])[b];
}

template <typename IdT, int THREADS>
struct PassSmem {
    uint64_t keys[RS_TILE];              // the tile's keys in output order
    uint64_t gofs[256];                  // output index of staged slot s of bin b = gofs[b] + s
    IdT ids[RS_TILE];                    // the ids, same order
    uint32_t whist[THREADS / 32][256];   // per-warp digit counts -> exclusive over the warps
    uint32_t binstart[256];              // first staged slot of every bin
    uint32_t wsum[8];
    uint32_t tile;
    uint8_t digit[RS_TILE];              // digit of every staged slot
};

// one stable pass on the digit (key >> shift) & 255.  THREADS = 256 (16 pairs per thread, 3 CTAs per SM with 32-bit ids) or 512
// (8 pairs per thread, 2 CTAs per SM): the tile is 4096 pairs either way; threads 0..255 own the bins.
template <typename IdT, bool WRITE_KEYS, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 512 ? 2 : (sizeof(IdT) == 4 ? 3 : 2))
k_radix_pass(const uint64_t* __restrict__ kin, const IdT* __restrict__ iin, uint64_t* __restrict__ kout, IdT* __restrict__ iout, uint64_t n,
             uint32_t shift, const uint64_t* __restrict__ bin_base, uint64_t* __restrict__ status, uint32_t* __restrict__ ticket, uint32_t tag) {
    constexpr int IPT = RS_TILE / THREADS;
    constexpr int WARPS = THREADS / 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PassSmem<IdT, THREADS>& S = *reinterpret_cast<PassSmem<IdT, THREADS>*>(smem_raw);

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) S.tile = atomicAdd(ticket, 1u);  // tiles in ticket order: every earlier tile is running or done
    for (uint32_t b = tid; b < WARPS * 256; b += THREADS) (&S.whist[0][0])[b] = 0;
    __syncthreads();
    const uint32_t tile = S.tile;
    const uint64_t tile_base = uint64_t(tile) * RS_TILE;
    const uint32_t tile_n = n - tile_base < uint64_t(RS_TILE) ? uint32_t(n - tile_base) : uint32_t(RS_TILE);
    const uint32_t first = warp * (32 * IPT) + lane;  // item j of this thread = tile slot first + 32 j (warp-striped)

    uint64_t key[IPT];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t li = first + 32 * j;
        key[j] = li < tile_n ? kin[tile_base + li] : ~uint64_t(0);
    }
    // rank of every item among the items of its warp with the same digit, in (item, lane) order.  The running count of a
    // digit is one shared-memory atomic by the first lane that holds it; the atomics of a warp are performed in program order,
    // and nothing waits for a result before all of them are on their way (the results are picked up in a second loop).
    uint32_t prevv[IPT];      // leader lanes: the digit's count before this item
    uint32_t lb[IPT / 2];     // per item: lanes below with the same digit (bits 0-7), the leader lane (bits 8-15)
    uint32_t* wh = S.whist[warp];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const bool valid = first + 32 * j < tile_n;
        const uint32_t d = valid ? uint32_t(key[j] >> shift) & 0xffu : 256u + lane;
        const uint32_t m = __match_any_sync(0xffffffffu, d);
        const uint32_t leader = uint32_t(__ffs(int(m)) - 1);
        prevv[j] = 0;
        if (valid && lane == leader) prevv[j] = atomicAdd(wh + d, uint32_t(__popc(m)));
        const uint32_t x = uint32_t(__popc(m & ((1u << lane) - 1u))) | (leader << 8);
        lb[j >> 1] = (j & 1) ? (lb[j >> 1] | (x << 16)) : x;
    }
    uint32_t rnk[IPT / 2];    // two 16-bit ranks per register
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t x = (j & 1) ? lb[j >> 1] >> 16 : lb[j >> 1] & 0xffffu;
        const uint32_t rk = __shfl_sync(0xffffffffu, prevv[j], int(x >> 8)) + (x & 0xffu);
        rnk[j >> 1] = (j & 1) ? (rnk[j >> 1] | (rk << 16)) : rk;
    }
    // the ids travel with the keys: asked for now, needed after the chained scan
    IdT idv[IPT];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t li = first + 32 * j;
        idv[j] = li < tile_n ? iin[tile_base + li] : IdT(0);
    }
    __syncthreads();

    // thread b < 256 owns bin b: counts exclusive over the warps, the tile's count published for the tiles behind
    const bool bin_thread = THREADS == 256 || tid < 256;  // (whole warps)
    uint32_t cnt = 0, incl = 0;
    uint64_t* st = status + uint64_t(tile) * 256 + tid;
    const uint64_t tagw = uint64_t(tag) << TAG_SHIFT;
    if (bin_thread) {
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const uint32_t t = S.whist[w][tid];
            S.whist[w][tid] = cnt;
            cnt += t;
        }
        st_status(st, tagw | (tile == 0 ? INCL_BIT : 0) | cnt);
        // first staged slot of the bin: exclusive scan of cnt over the bins
        incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= uint32_t(o)) incl += t;
        }
        if (lane == 31) S.wsum[warp] = incl;
    }
    __syncthreads();
    if (bin_thread) {
        uint32_t wbase = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) wbase += uint32_t(w) < warp ? S.wsum[w] : 0u;
        const uint32_t binstart = wbase + incl - cnt;
        S.binstart[tid] = binstart;
        // chained scan: pairs of this bin in all earlier tiles
        uint64_t excl = 0;
        if (tile > 0) {
            int64_t t = int64_t(tile) - 1;
            for (bool open = true; open;) {
                // four earlier tiles asked for together (one round trip), taken in order
                uint64_t wv[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) wv[q] = t - q >= 0 ? ld_status(status + uint64_t(t - q) * 256 + tid) : 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (open && t - q >= 0) {
                        uint64_t x = wv[q];
                        while ((x >> TAG_SHIFT) != tag) x = ld_status(status + uint64_t(t - q) * 256 + tid);
                        excl += x & CNT_MASK;
                        if (x & INCL_BIT) open = false;
                    }
                }
                t -= 4;
            }
            st_status(st, tagw | INCL_BIT | (excl + cnt));
        }
        S.gofs[tid] = bin_base[tid] + excl - binstart;
    }
    __syncthreads();

    // pairs into output order (shared), then out as one coalesced run per bin
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        if (first + 32 * j < tile_n) {
            const uint32_t d = uint32_t(key[j] >> shift) & 0xffu;
            const uint32_t rk = (j & 1) ? rnk[j >> 1] >> 16 : rnk[j >> 1] & 0xffffu;
            const uint32_t slot = S.binstart[d] + S.whist[warp][d] + rk;
            S.digit[slot] = uint8_t(d);
            if (WRITE_KEYS) S.keys[slot] = key[j];
            S.ids[slot] = idv[j];
        }
    }
    __syncthreads();
    if (tile_n == uint32_t(RS_TILE)) {
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t i = tid + uint32_t(j) * THREADS;
            const uint64_t g = S.gofs[S.digit[i]] + i;
            if (WRITE_KEYS) kout[g] = S.keys[i];
            iout[g] = S.ids[i];
        }
    } else {
        for (uint32_t i = tid; i < tile_n; i += THREADS) {
            const uint64_t g = S.gofs[S.digit[i]] + i;
            if (WRITE_KEYS) kout[g] = S.keys[i];
            iout[g] = S.ids[i];
        }
    }
}

// one thread per record; the previous record's key words come from the lane below (lane 0 fetches them itself)
template <typename IdT>
__global__ void k_egsa_finish(ReadsView v, const uint64_t* __restrict__ packed, const IdT* __restrict__ ids, uint64_t n,
                              uint32_t* __restrict__ lcp, uint32_t* __restrict__ text, uint32_t* __restrict__ suff,
                              uint8_t* __restrict__ bwt, uint64_t before) {
    // before: the record that precedes record 0 in the whole index, text << 32 | suff (a key range that does not start the
    // index); ~0 = none, lcp[0] = 0
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;  // blockDim.x is a multiple of 32: whole warps leave together
    const uint32_t lane = threadIdx.x & 31;
    const bool valid = i < n;
    uint64_t r = 0, st = 0;
    uint32_t p = 0, len = 0;
    if (valid) {
        v.decode(ids[i], r, p);
        st = v.start(r);
        len = v.len(r);
        text[i] = uint32_t(r);
        suff[i] = p;
        bwt[i] = p ? v.bases[st + p - 1] : uint8_t('$');
    }
    const uint64_t* row = packed + v.row(r, st);
    const uint32_t la = len - p;
    // the record before: the lane below's, or fetched (first lane of a warp)
    uint32_t lb = __shfl_up_sync(0xffffffffu, la, 1);
    const uint64_t* row0 = row;
    uint32_t p0 = 0, len0 = 0;
    const bool has_prev = valid && (i > 0 || before != ~uint64_t(0));
    const bool fetch = lane == 0 && has_prev;
    if (fetch) {
        uint64_t r0;
        if (i > 0) {
            v.decode(ids[i - 1], r0, p0);
        } else {
            r0 = before >> 32;
            p0 = uint32_t(before);
        }
        const uint64_t st0 = v.start(r0);
        len0 = v.len(r0);
        row0 = packed + v.row(r0, st0);
        lb = len0 - p0;
    }
    uint32_t l = has_prev ? (la < lb ? la : lb) : 0;  // the shorter of the two suffixes
    bool open = l > 0;
    for (uint32_t w = 0; __any_sync(0xffffffffu, open && 32 * w < l); ++w) {
        const uint64_t mine = valid ? suffix_word(row, len, p, w) : 0;
        uint64_t prev = __shfl_up_sync(0xffffffffu, mine, 1);
        if (fetch) prev = suffix_word(row0, len0, p0, w);
        if (open && 32 * w < l) {
            const uint64_t x = prev ^ mine;
            if (x) {
                const uint32_t d = 32 * w + uint32_t(__clzll(static_cast<long long>(x))) / 2;
                l = d < l ? d : l;
                open = false;
            }
        }
    }
    if (valid) lcp[i] = l;
}

// ---- one key range of the index ---------------------------------------------------------------------------------------------
// The suffixes whose first key word (32 symbols, zero padded) lies in [lo, hi) are a contiguous range of the index: a GPU that
// cannot hold the scratch of the whole collection, or one GPU of several, sorts only those.  Two sweeps over all suffix slots: count
// per chunk of 4096 slots (+ how many lie below the range, + the selected per length), then a stable compaction of their ids.
//   equal lengths: slot i = suffix id i (the iota, length i / R): the ids go to both id buffers, already shortest first.
//   ragged:        slot i = suffix (r, p) with start_r + r + p = i, the (read, offset) order of k_init_ids_ragged.  A CTA finds the
//                  reads its chunk touches (two binary searches over the device offsets), stages their slot starts in shared memory,
//                  and every thread finds its first read there and walks forward.  The ids (r << shift) | p go to one buffer; the
//                  length pass then brings them to shortest-first order as in the whole build.
constexpr int SEL_THREADS = 256;
constexpr int SEL_IPT = 16;
constexpr int SEL_CHUNK = SEL_THREADS * SEL_IPT;
constexpr uint32_t SEL_HIST_BINS = 2048;  // ragged: per-CTA length histogram in shared memory while L + 1 bins fit, else global atomics

struct SelStats {
    unsigned long long n_below;   // suffixes whose first key word is below lo = index position of the range's first record
    unsigned long long n_sel;
};

// ragged: the last read r with start_r + r <= i (the read that owns slot i)
__device__ __forceinline__ uint64_t read_of_slot(const uint64_t* __restrict__ off, uint64_t R, uint64_t i) {
    uint64_t a = 0, b = R;  // off[a] + a <= i < off[b] + b
    while (b - a > 1) {
        const uint64_t m = a + ((b - a) >> 1);
        if (off[m] + m <= i) a = m;
        else b = m;
    }
    return a;
}

template <typename IdT, bool WRITE, bool RAGGED>
__global__ void __launch_bounds__(SEL_THREADS) k_range_select(ReadsView v, const uint64_t* __restrict__ packed, uint64_t n, uint64_t lo, uint64_t hi,
                                                              uint64_t* __restrict__ chunk_cnt, unsigned long long* __restrict__ len_hist,
                                                              SelStats* __restrict__ stats, IdT* __restrict__ out0, IdT* __restrict__ out1) {
    __shared__ uint32_t s_w[SEL_THREADS / 32];
    __shared__ uint32_t s_below, s_first_len_cnt;
    // ragged: slot starts of the chunk's reads r0 + k relative to r0's (k <= SEL_CHUNK: every read after r0 owns a slot of the
    // chunk), and the chunk's length histogram
    __shared__ uint32_t s_start[RAGGED ? SEL_CHUNK + 1 : 1];
    __shared__ uint32_t s_hist[RAGGED && !WRITE ? SEL_HIST_BINS : 1];
    __shared__ uint64_t s_r[3];  // ragged: r0 = the read of the chunk's first slot, r1 = of its last, off[r0]
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t chunk_base = uint64_t(blockIdx.x) * SEL_CHUNK;
    const uint64_t base = chunk_base + uint64_t(tid) * SEL_IPT;
    const uint64_t first_len = RAGGED ? 0 : chunk_base / v.R;  // equal lengths: the length of the chunk's first suffix
    const bool shared_hist = RAGGED && !WRITE && v.L < SEL_HIST_BINS;
    if (tid == 0) { s_below = 0; s_first_len_cnt = 0; }
    if (RAGGED) {
        if (tid == 0) {
            s_r[0] = read_of_slot(v.off, v.R, chunk_base);
            s_r[2] = v.off[s_r[0]];
        }
        if (tid == 32) s_r[1] = read_of_slot(v.off, v.R, (chunk_base + SEL_CHUNK < n ? chunk_base + SEL_CHUNK : n) - 1);
        if (shared_hist)
            for (uint32_t b = tid; b <= v.L; b += SEL_THREADS) s_hist[b] = 0;
        __syncthreads();
        const uint64_t r0 = s_r[0], st0 = s_r[2] + r0;
        const uint32_t nr = uint32_t(s_r[1] - r0) + 2;  // reads r0 .. r1 and the start of the one after
        for (uint32_t k = tid; k < nr; k += SEL_THREADS) s_start[k] = uint32_t(v.off[r0 + k] + r0 + k - st0);
    }
    __syncthreads();
    // the thread's first slot: read r = r0 + k, offset p, length len, bases from st
    uint64_t r = 0, st = 0;
    uint32_t k = 0, p = 0, len = v.L;
    const uint64_t r0 = RAGGED ? s_r[0] : 0;
    if (RAGGED && base < n) {
        const uint32_t b = uint32_t(base - (s_r[2] + r0));
        uint32_t a = 0, z = uint32_t(s_r[1] - r0) + 1;  // s_start[a] <= b < s_start[z]
        while (z - a > 1) {
            const uint32_t m = (a + z) >> 1;
            if (s_start[m] <= b) a = m;
            else z = m;
        }
        k = a;
        p = b - s_start[k];
        len = s_start[k + 1] - s_start[k] - 1;
        r = r0 + k;
        st = s_r[2] + s_start[k] - k;
    }
    const uint32_t k_first = k, p_first = p;
    uint32_t sel = 0, below = 0, at_first_len = 0;
#pragma unroll 4
    for (int j = 0; j < SEL_IPT; ++j) {
        const uint64_t i = base + j;
        if (i < n) {
            uint32_t q;
            if (RAGGED) {
                if (p > len) {  // past read r's terminator: the next read (every read owns at least its terminator slot)
                    ++k;
                    p = 0;
                    len = s_start[k + 1] - s_start[k] - 1;
                    r = r0 + k;
                    st += (s_start[k] - s_start[k - 1]) - 1;
                }
                q = p++;
            } else {
                v.decode(IdT(i), r, q);
                st = v.start(r);
            }
            const uint64_t key = suffix_word(packed + v.row(r, st), len, q, 0);
            if (key < lo) ++below;
            else if (hi == 0 || key < hi) {
                sel |= 1u << j;
                if (!WRITE) {
                    const uint32_t sl = len - q;
                    if (RAGGED) {
                        if (shared_hist) atomicAdd(&s_hist[sl], 1u);
                        else atomicAdd(len_hist + sl, 1ull);
                    } else if (sl == first_len) {
                        ++at_first_len;
                    } else {
                        atomicAdd(len_hist + sl, 1ull);  // (a chunk seldom spans two lengths)
                    }
                }
            }
        }
    }
    const uint32_t cnt = uint32_t(__popc(sel));
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= uint32_t(o)) inc += t;
    }
    if (lane == 31) s_w[warp] = inc;
    if (!WRITE) {
        const uint32_t wb = __reduce_add_sync(0xffffffffu, below), wf = __reduce_add_sync(0xffffffffu, at_first_len);
        if (lane == 0 && wb) atomicAdd(&s_below, wb);
        if (lane == 0 && wf) atomicAdd(&s_first_len_cnt, wf);
    }
    __syncthreads();
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < SEL_THREADS / 32; ++w) {
        wbase += uint32_t(w) < warp ? s_w[w] : 0u;
        total += s_w[w];
    }
    if (!WRITE) {
        if (tid == 0) {
            chunk_cnt[blockIdx.x] = total;
            if (s_below) atomicAdd(&stats->n_below, (unsigned long long)s_below);
            if (total) atomicAdd(&stats->n_sel, (unsigned long long)total);
            if (s_first_len_cnt) atomicAdd(len_hist + first_len, (unsigned long long)s_first_len_cnt);
        }
        if (shared_hist)
            for (uint32_t b = tid; b <= v.L; b += SEL_THREADS)
                if (s_hist[b]) atomicAdd(len_hist + b, (unsigned long long)s_hist[b]);
    } else {
        uint64_t at = chunk_cnt[blockIdx.x] + wbase + inc - cnt;
        if (RAGGED) {  // the same walk again, ids in (read, offset) order
            k = k_first;
            p = p_first;
            len = s_start[k + 1] - s_start[k] - 1;
            for (int j = 0; j < SEL_IPT && sel >> j; ++j) {
                if (p > len) {
                    ++k;
                    p = 0;
                    len = s_start[k + 1] - s_start[k] - 1;
                }
                if (sel & (1u << j)) out0[at++] = IdT(((r0 + k) << v.shift) | p);
                ++p;
            }
        } else {
#pragma unroll 4
            for (int j = 0; j < SEL_IPT; ++j)
                if (sel & (1u << j)) {
                    out0[at] = IdT(base + j);
                    out1[at] = IdT(base + j);
                    ++at;
                }
        }
    }
}

// in-place exclusive scan of cnt[0 .. nb) by one CTA
__global__ void __launch_bounds__(1024) k_scan_chunks(uint64_t* __restrict__ cnt, uint64_t nb) {
    __shared__ uint64_t s_part[1024];
    const uint64_t per = (nb + 1023) / 1024;
    const uint64_t a = uint64_t(threadIdx.x) * per, b = a + per < nb ? a + per : nb;
    uint64_t sum = 0;
    for (uint64_t i = a; i < b; ++i) sum += cnt[i];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t run = 0;
        for (int t = 0; t < 1024; ++t) {
            const uint64_t x = s_part[t];
            s_part[t] = run;
            run += x;
        }
    }
    __syncthreads();
    uint64_t run = s_part[threadIdx.x];
    for (uint64_t i = a; i < b; ++i) {
        const uint64_t x = cnt[i];
        cnt[i] = run;
        run += x;
    }
}

struct KeyRange {              // host side: one key range of the index
    uint64_t lo, hi;           // first key word in [lo, hi); hi == 0: no upper bound
    uint64_t cap;              // records the output arrays hold
    uint64_t before;           // the record before the range, text << 32 | suff; ~0 = none / not known
    uint64_t n_out, first_out; // results: records written, index position of the first one
};

inline unsigned blocks_for(uint64_t n, int t) { return unsigned((n + uint64_t(t) - 1) / uint64_t(t)); }

template <typename IdT>
cudaError_t build_typed(ReadsView v, uint64_t n_all, uint64_t total_bases, const uint64_t* n_le_all, KeyRange* range, uint32_t* d_lcp,
                        uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, cudaStream_t stream, uint64_t* launches) {
    const uint32_t W = (v.L + 31) / 32;
    uint64_t n = n_all;                // suffixes this call sorts (a key range: known after the first sweep)
    const uint64_t* n_le = n_le_all;
    std::vector<uint64_t> n_le_sel;
    uint64_t tiles = (n + RS_TILE - 1) / RS_TILE;
    const uint32_t len_places = v.shift ? (v.L >= 256 ? 2u : 1u) : 0u;
    uint32_t passes = len_places;
    for (uint32_t w = 0; w < W; ++w) {
        const uint32_t syms = v.L - 32 * w < 32 ? v.L - 32 * w : 32;
        passes += (2 * syms + 7) / 8;
    }
    if (passes >= (1u << (64 - TAG_SHIFT)) - 1u || tiles >= (uint64_t(1) << 31)) return cudaErrorInvalidConfiguration;
    const uint64_t packed_words = (total_bases >> 5) + 2 * v.R + 2;
    uint64_t *packed = nullptr, *k0 = nullptr, *k1 = nullptr, *status = nullptr, *misc = nullptr, *chunk_cnt = nullptr, *sel_misc = nullptr;
    IdT *i0 = nullptr, *i1 = nullptr;
    uint32_t* tickets = nullptr;
    cudaError_t e = cudaSuccess;
    auto done = [&](cudaError_t rc) {
        cudaFree(packed); cudaFree(k0); cudaFree(k1); cudaFree(i0); cudaFree(i1); cudaFree(status); cudaFree(misc); cudaFree(tickets);
        cudaFree(chunk_cnt); cudaFree(sel_misc);
        return rc;
    };
    // misc: hist[8][256] | bin_base[8][256] | bad flag
    const size_t misc_bytes = size_t(2 * MAX_PLACES * 256 + 1) * 8;
    if ((e = cudaMalloc(reinterpret_cast<void**>(&misc), misc_bytes)) != cudaSuccess) return done(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&tickets), size_t(passes + 1) * 4)) != cudaSuccess) return done(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&packed), packed_words * 8)) != cudaSuccess) return done(e);
    if ((e = cudaMemsetAsync(misc, 0, misc_bytes, stream)) != cudaSuccess) return done(e);
    if ((e = cudaMemsetAsync(tickets, 0, size_t(passes + 1) * 4, stream)) != cudaSuccess) return done(e);
    unsigned long long* hist = reinterpret_cast<unsigned long long*>(misc);
    uint64_t* bin_base = misc + MAX_PLACES * 256;
    uint32_t* d_bad = reinterpret_cast<uint32_t*>(misc + 2 * MAX_PLACES * 256);

    k_pack_reads<<<blocks_for(v.R * 32, 256), 256, 0, stream>>>(v, packed, d_bad);
    *launches += 1;
    {   // a base outside ACGT / acgt has no 2-bit code: refuse before sorting instead of building a wrong index
        uint32_t h_bad = 0;
        if ((e = cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return done(e);
        if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return done(e);
        if (h_bad) return done(cudaErrorInvalidValue);
    }
    const uint64_t n_chunks = (n_all + SEL_CHUNK - 1) / SEL_CHUNK;
    if (range) {  // first sweep: who is in the range
        if (n_chunks >= (uint64_t(1) << 31)) return done(cudaErrorInvalidConfiguration);
        const size_t sel_bytes = (size_t(v.L) + 1) * 8 + sizeof(SelStats);
        if ((e = cudaMalloc(reinterpret_cast<void**>(&chunk_cnt), n_chunks * 8)) != cudaSuccess) return done(e);
        if ((e = cudaMalloc(reinterpret_cast<void**>(&sel_misc), sel_bytes)) != cudaSuccess) return done(e);
        if ((e = cudaMemsetAsync(sel_misc, 0, sel_bytes, stream)) != cudaSuccess) return done(e);
        unsigned long long* len_hist = reinterpret_cast<unsigned long long*>(sel_misc);
        SelStats* stats = reinterpret_cast<SelStats*>(sel_misc + v.L + 1);
        if (v.shift) k_range_select<IdT, false, true><<<unsigned(n_chunks), SEL_THREADS, 0, stream>>>(v, packed, n_all, range->lo, range->hi, chunk_cnt,
                                                                                                      len_hist, stats, nullptr, nullptr);
        else k_range_select<IdT, false, false><<<unsigned(n_chunks), SEL_THREADS, 0, stream>>>(v, packed, n_all, range->lo, range->hi, chunk_cnt,
                                                                                                len_hist, stats, nullptr, nullptr);
        k_scan_chunks<<<1, 1024, 0, stream>>>(chunk_cnt, n_chunks);
        *launches += 2;
        std::vector<uint64_t> h(size_t(v.L) + 1 + sizeof(SelStats) / 8);
        if ((e = cudaMemcpyAsync(h.data(), sel_misc, sel_bytes, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return done(e);
        if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return done(e);
        range->first_out = h[size_t(v.L) + 1];
        n = h[size_t(v.L) + 2];
        range->n_out = n;
        if (n > range->cap) return done(cudaErrorInvalidPitchValue);  // (the caller's arrays are too small: n_out says by how much)
        if (n == 0) return done(cudaSuccess);
        n_le_sel.assign(size_t(v.L) + 1, 0);
        for (uint32_t t = 0; t <= v.L; ++t) n_le_sel[t] = (t ? n_le_sel[t - 1] : 0) + h[t];
        n_le = n_le_sel.data();
        tiles = (n + RS_TILE - 1) / RS_TILE;
    }
    if ((e = cudaMalloc(reinterpret_cast<void**>(&status), tiles * 256 * 8)) != cudaSuccess) return done(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&k0), n * 8)) != cudaSuccess) return done(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&k1), n * 8)) != cudaSuccess) return done(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&i0), n * sizeof(IdT))) != cudaSuccess) return done(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&i1), n * sizeof(IdT))) != cudaSuccess) return done(e);
    if ((e = cudaMemsetAsync(status, 0, tiles * 256 * 8, stream)) != cudaSuccess) return done(e);  // tag 0 = no pass
    if (range && v.shift) {  // second sweep, ragged: the selected ids in (read, offset) order, sorted by length below
        k_range_select<IdT, true, true><<<unsigned(n_chunks), SEL_THREADS, 0, stream>>>(v, packed, n_all, range->lo, range->hi, chunk_cnt, nullptr, nullptr,
                                                                                        i0, nullptr);
        *launches += 1;
    } else if (range) {  // second sweep, equal lengths: the selected ids in id order (= shortest first, then read id), into both buffers
        k_range_select<IdT, true, false><<<unsigned(n_chunks), SEL_THREADS, 0, stream>>>(v, packed, n_all, range->lo, range->hi, chunk_cnt, nullptr, nullptr,
                                                                                         i0, i1);
        *launches += 1;
    } else if (v.shift) {
        k_init_ids_ragged<IdT><<<blocks_for(v.R * 32, 256), 256, 0, stream>>>(v, i0);
        *launches += 1;
    } else {  // both buffers: a word's passes leave the suffixes that are too short for it where they are, in either buffer
        k_init_ids_equal<IdT><<<blocks_for(n, 256), 256, 0, stream>>>(i0, n);
        k_init_ids_equal<IdT><<<blocks_for(n, 256), 256, 0, stream>>>(i1, n);
        *launches += 2;
    }

    uint64_t *kc = k0, *ka = k1;  // current / alternate
    IdT *ic = i0, *ia = i1;
    uint32_t seq = 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // 256 threads x 16 pairs (3 CTAs per SM at 80 registers with 32-bit ids, 2 at 128 with 64-bit ids) or 512 threads x 8 pairs (2 CTAs
    // per SM at 64 registers).  Measured on the C2-size index: 32-bit ids 128 ms / 139 ms, 64-bit ids 151 ms / 146 ms -- the default is
    // the faster one of each; E2S_RADIX_THREADS overrides (tests run both).
    int rs_threads = sizeof(IdT) == 4 ? 256 : 512;
    if (const char* t = getenv("E2S_RADIX_THREADS")) rs_threads = atoi(t) == 512 ? 512 : 256;
    const int smem_bytes = rs_threads == 512 ? int(sizeof(PassSmem<IdT, 512>)) : int(sizeof(PassSmem<IdT, 256>));
    if ((e = cudaFuncSetAttribute(k_radix_pass<IdT, true, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(PassSmem<IdT, 256>)))) != cudaSuccess) return done(e);
    if ((e = cudaFuncSetAttribute(k_radix_pass<IdT, false, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(PassSmem<IdT, 256>)))) != cudaSuccess) return done(e);
    if ((e = cudaFuncSetAttribute(k_radix_pass<IdT, true, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(PassSmem<IdT, 512>)))) != cudaSuccess) return done(e);
    if ((e = cudaFuncSetAttribute(k_radix_pass<IdT, false, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(PassSmem<IdT, 512>)))) != cudaSuccess) return done(e);
    // Sorts the current order on `places` digit places of key word w (w_base = 32 w symbols before it; LEN_WORD: the length
    // key, everything moves).  n_le[t] = suffixes of t symbols or fewer.  A suffix that ends before the symbols of a place has
    // digit 0 there and is still where the shortest-first order put it (a prefix of the current order, identical in both
    // buffers): place j moves only the suffixes longer than that, [first_j, n).
    auto sort_word = [&](uint32_t w, uint32_t begin_bit, uint32_t places) {
        uint64_t first_of[MAX_PLACES];
        for (uint32_t j = 0; j < places; ++j) {
            if (w == LEN_WORD) { first_of[j] = 0; continue; }
            const int s_lo = 28 - int(begin_bit / 2) - 4 * int(j);  // first symbol of the word that place j holds
            const uint64_t t = uint64_t(32) * w + uint64_t(s_lo > 0 ? s_lo : 0);
            first_of[j] = n_le[t < v.L ? t : v.L];
        }
        const uint64_t first = first_of[places - 1];  // the widest range: what the word's keys are made for
        const uint64_t m = n - first;
        if (m == 0) return;  // (a key range whose suffixes are all too short for the word)
        PlaceSkip skip;
        for (uint32_t j = 0; j < MAX_PLACES; ++j) skip.n[j] = j < places ? first_of[j] - first : 0;
        const uint64_t hist_blocks_want = (m + 255) / 256;
        const unsigned hist_blocks = unsigned(hist_blocks_want < uint64_t(sms) * 8 ? hist_blocks_want : uint64_t(sms) * 8);
        k_keys_hist<IdT><<<hist_blocks, 256, 0, stream>>>(v, packed, ic + first, m, w, begin_bit, places, kc + first, ka + first,
                                                          first_of[0] - first, hist);
        k_scan_hist<<<1, 256, 0, stream>>>(hist, bin_base, skip);
        *launches += 2;
        for (uint32_t j = 0; j < places; ++j, ++seq) {
            const uint32_t sh = begin_bit + 8 * j;
            const uint64_t f = first_of[j], mj = n - f;
            if (mj == 0) continue;  // nothing long enough for this place: no pass, the current buffers stay current
            const unsigned tiles_j = unsigned((mj + RS_TILE - 1) / RS_TILE);
            const bool wk = j + 1 < places;  // the keys of a word are not looked at again after its last place
            if (rs_threads == 512) {
                if (wk) k_radix_pass<IdT, true, 512><<<tiles_j, 512, smem_bytes, stream>>>(kc + f, ic + f, ka + f, ia + f, mj, sh, bin_base + 256 * j, status, tickets + seq, seq + 1);
                else k_radix_pass<IdT, false, 512><<<tiles_j, 512, smem_bytes, stream>>>(kc + f, ic + f, ka + f, ia + f, mj, sh, bin_base + 256 * j, status, tickets + seq, seq + 1);
            } else {
                if (wk) k_radix_pass<IdT, true, 256><<<tiles_j, 256, smem_bytes, stream>>>(kc + f, ic + f, ka + f, ia + f, mj, sh, bin_base + 256 * j, status, tickets + seq, seq + 1);
                else k_radix_pass<IdT, false, 256><<<tiles_j, 256, smem_bytes, stream>>>(kc + f, ic + f, ka + f, ia + f, mj, sh, bin_base + 256 * j, status, tickets + seq, seq + 1);
            }
            *launches += 1;
            uint64_t* tk = kc; kc = ka; ka = tk;
            IdT* ti = ic; ic = ia; ia = ti;
        }
    };
    if (len_places) {  // ragged: shortest first, then both buffers hold that order
        sort_word(LEN_WORD, 0, len_places);
        if ((e = cudaMemcpyAsync(ia, ic, n * sizeof(IdT), cudaMemcpyDeviceToDevice, stream)) != cudaSuccess) return done(e);
    }
    for (int w = int(W) - 1; w >= 0; --w) {
        // symbols of this word that exist in the longest suffix: only those bits can differ
        const uint32_t syms = v.L - 32 * uint32_t(w) < 32 ? v.L - 32 * uint32_t(w) : 32;
        sort_word(uint32_t(w), 64 - 2 * syms, (2 * syms + 7) / 8);
    }
    k_egsa_finish<IdT><<<blocks_for(n, 256), 256, 0, stream>>>(v, packed, ic, n, d_lcp, d_text, d_suff, d_bwt, range ? range->before : ~uint64_t(0));
    *launches += 1;
    if ((e = cudaGetLastError()) != cudaSuccess) return done(e);
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return done(e);
    return done(cudaSuccess);
}

// ragged ids (r << shift) | p: the bits of p in [0, L]
inline uint32_t ragged_shift(uint32_t L) {
    uint32_t bits = 1;
    while ((L >> bits) != 0) ++bits;
    return bits;
}

}  // namespace

// d_off == nullptr: R reads of L bases each; else R + 1 DEVICE offsets (h_off = the same on the host), L = the longest read,
// total_bases = off[R].
// scratch (freed before returning): two key buffers + two id buffers + tile status = 24.5 (32-bit ids) / 32.5 bytes per suffix
cudaError_t build_egsa(const uint8_t* d_reads, const uint64_t* d_off, const uint64_t* h_off, uint64_t R, uint32_t L, uint64_t total_bases,
                       uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, cudaStream_t stream, uint64_t* launches) {
    ReadsView v;
    v.bases = d_reads;
    v.off = d_off;
    v.R = R;
    v.L = L;
    v.shift = 0;
    const uint64_t n = total_bases + R;
    std::vector<uint64_t> n_le(size_t(L) + 1, 0);  // n_le[t] = suffixes of t symbols or fewer
    bool wide;
    if (d_off) {
        if (L >= 65536 || !h_off) return cudaErrorInvalidConfiguration;
        v.shift = ragged_shift(L);
        wide = R > (uint64_t(1) << (32 - v.shift));
        std::vector<uint64_t> at_least(size_t(L) + 2, 0);  // reads of t bases or more
        for (uint64_t r = 0; r < R; ++r) ++at_least[size_t(h_off[r + 1] - h_off[r])];
        for (uint32_t t = L; t-- > 0;) at_least[t] += at_least[t + 1];
        n_le[0] = R;
        for (uint32_t t = 1; t <= L; ++t) n_le[t] = n_le[t - 1] + at_least[t];
    } else {
        wide = n > 0xffffffffull;
        for (uint32_t t = 0; t <= L; ++t) n_le[t] = R * (uint64_t(t) + 1);
    }
    if (getenv("E2S_BUILD_IDS64")) wide = true;  // test hook: the 64-bit instantiation on small inputs
    return wide ? build_typed<uint64_t>(v, n, total_bases, n_le.data(), nullptr, d_lcp, d_text, d_suff, d_bwt, stream, launches)
                : build_typed<uint32_t>(v, n, total_bases, n_le.data(), nullptr, d_lcp, d_text, d_suff, d_bwt, stream, launches);
}

// One key range of the index: the records of the suffixes whose first key word (32 symbols at 2 bits, A=0 C=1 G=2 T=3, most
// significant first, zero padded) lies in [key_lo, key_hi) (key_hi == 0: no upper bound) -- a contiguous range of the index,
// *first_out = the index position of its first record, *n_out = how many there are (also set when they exceed `cap`:
// cudaErrorInvalidPitchValue, nothing written).  before = the record that precedes the range (text << 32 | suff) for lcp[0], ~0 =
// none / not known (lcp[0] = 0).  d_off == nullptr: R reads of L bases each; else R + 1 DEVICE offsets, L = the longest read,
// total_bases = off[R].  The id width is the whole collection's, as in build_egsa.  Scratch: 24.5 / 32.5 bytes per suffix OF THE
// RANGE + 8 bytes per 4096 suffixes of the collection.
cudaError_t build_egsa_range(const uint8_t* d_reads, const uint64_t* d_off, uint64_t R, uint32_t L, uint64_t total_bases, uint64_t key_lo,
                             uint64_t key_hi, uint64_t before, uint64_t cap, uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt,
                             uint64_t* n_out, uint64_t* first_out, cudaStream_t stream, uint64_t* launches) {
    ReadsView v;
    v.bases = d_reads;
    v.off = d_off;
    v.R = R;
    v.L = L;
    v.shift = 0;
    const uint64_t n = total_bases + R;
    bool wide = n > 0xffffffffull;
    if (d_off) {
        if (L >= 65536) return cudaErrorInvalidConfiguration;
        v.shift = ragged_shift(L);
        wide = R > (uint64_t(1) << (32 - v.shift));
    }
    if (getenv("E2S_BUILD_IDS64")) wide = true;
    KeyRange range{key_lo, key_hi, cap, before, 0, 0};
    // (the suffix lengths of a range come from its selection sweep: no whole-collection n_le)
    const cudaError_t e = wide ? build_typed<uint64_t>(v, n, total_bases, nullptr, &range, d_lcp, d_text, d_suff, d_bwt, stream, launches)
                               : build_typed<uint32_t>(v, n, total_bases, nullptr, &range, d_lcp, d_text, d_suff, d_bwt, stream, launches);
    *n_out = range.n_out;
    *first_out = range.first_out;
    return e;
}

}  // namespace e2s
