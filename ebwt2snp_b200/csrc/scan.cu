// Phase 1 (ebwt2clust) in ONE pass over the resident bit-sliced LCP: k_cluster_scan.
//
// cluster_lm / append_entry (ref:ebwt2clust.cpp:54-139) in their stencil form (cluster.cu, SURVEY.md 8(a) A2).  The
// kernel reads one byte per position once, keeps the START / END bit masks in REGISTERS (they are never written to
// global memory), and goes straight on to the records.
//
//   input     the LCP as the loads left it for this kernel (k_derive, unpack.cu): bit-sliced, plane-major in blocks of
//             2048 positions -- block b = eight runs of 32 words, run p = bit plane p of the LCP value (<= 127) for
//             p < 7 and the plane A (bit x = lcp[x-1] > lcp[x]) for p = 7, word g of a run = the 64 positions
//             2048 b + 64 g ...  Nothing in it depends on an option of either tool.  "lcp >= k" is then a bit-sliced
//             comparator: one LOP3 per plane word ((k_b ? ~x | lt : ~x & lt) as a single 3-input function), 14 logic
//             instructions for 64 positions instead of the 64+ of a byte-wise compare; the local-minimum test of the
//             stencil is A & ~(A >> 1).  A warp reads a run with one conflict-free 8-byte load per lane at a constant
//             offset from its base: no address arithmetic.
//   tiles     16 384 positions = 8 blocks = one per warp.  One CTA per CHUNK of consecutive tiles, no communication
//             between CTAs; SC_STAGES tiles in flight per CTA: one bulk copy of the tile's 16 KB, two 128-byte tensor
//             boxes with the plane words of the group before and of the group after the tile, and (fused prefilter) one
//             bulk copy of the tile's window of the base-code bit planes, all signalling the same mbarrier.
//   masks     each thread owns 64 consecutive positions = one 64-bit word per mask (G, A -> END, START); the G / A bits of
//             the position before and after them come from the neighbouring words of the same runs.
//   ranks     kept ENDs (K = E minus the ENDs of clusters shorter than min_len, a bit-parallel function of the masks: a
//             START at most min_len - 2 positions before, min_len <= 33) are ranked by ONE block scan; each thread
//             scatters the tile-local positions of its kept ENDs to a shared list -- nothing else happens at lane
//             efficiency popcount / max popcount.
//   records   one lane per list entry (dense): nearest START at or before the END from the tile's START words in shared
//             memory (own word, else the per-warp ballots of non-empty words point at the word), length mod 2^16, stores
//             (start u64, len u16) in position order into the chunk's segment, length histogram + n_bases of
//             statistics() (ref:clust2snp.cpp:899-907), and -- fused mode -- the BWT prefilter of find_variants
//             (ref:clust2snp.cpp:402-429) as the one-popcount bound of planes.cuh on the plane window; the survivors are
//             appended to the list K3x reads.
//   state     the open-cluster state and the record count are carried from tile to tile by warp 0.  What a chunk cannot
//             know -- whether a cluster is open when it starts -- only matters for its first event: if that is an END
//             ("head" of the chunk) the record is left to k_chunk_resolve, which sees all chunks' summaries.  The only
//             END of a tile whose START is not in the tile is its first event ("carried" END): warp 0 tests it exactly,
//             wrapped 16-bit length included (a tile is shorter than 65 503 positions, so no other END can wrap).
//   barriers  two per tile: (A) after the masks, (B) after the scatter; the START words are double buffered by tile parity.
//
// Algorithmic bytes: 1 B/position read + 10 B per written record (+ 0.25 B per position inside analysed clusters of
// base-code planes in fused mode).
// Not handled here (callers fall back to k_lcp_flags + k_cluster_emit): min_len > 33, shards with an LCP value > 127.

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "common.cuh"
#include "internal.h"
#include "planes.cuh"

namespace e2s {

namespace {

constexpr uint32_t FULL = 0xffffffffu;
constexpr int SC_THREADS = 256;
constexpr int SC_WARPS = SC_THREADS / 32;
constexpr int SC_V = 64;                       // positions per thread = one word per plane
constexpr int SC_T = SC_THREADS * SC_V;        // 16384 positions per tile = SC_WARPS blocks of LCPT_BLOCK positions
constexpr int SC_EDGE = 128;                   // bytes of an edge box: 8 plane runs x 2 words
constexpr int SC_STAGE_BYTES = SC_T + 2 * SC_EDGE;  // the tile, the box before it, the box after it
constexpr int SC_STAGES = 2;                   // LCP tiles in flight / being read per CTA (a stage is free once its words are in registers)
constexpr int SC_OCC = 4;                      // resident CTAs per SM the register / shared-memory budget is sized for
constexpr int SC_PSLOTS = SC_STAGES + 1;       // plane windows: a window is read until its tile's records are written, after the stage was refilled
constexpr int SC_PF_QUADS = SC_T / 64 + PL_PAD / 64;  // plane quads of one tile and of the PL_PAD positions before it
constexpr int SC_PF_BYTES = SC_PF_QUADS * 16;  // 4144
constexpr int SC_PF_STRIDE = 4224;             // slot stride (128-byte multiple)
constexpr int SC_DYN_SMEM = SC_STAGES * SC_STAGE_BYTES + SC_PSLOTS * SC_PF_STRIDE;
constexpr int SC_CAP = 512;                    // kept ENDs per list window (a typical tile lists ~300)
static_assert(SC_STAGES == 2, "stage = tile parity");
static_assert(LCPT_BLOCK == 32 * SC_V && SC_T == SC_WARPS * LCPT_BLOCK, "one block of the bit-sliced LCP per warp");
static_assert(SC_T <= (1 << 14), "tile-local positions fit 14 bits");

// open-cluster state (as in cluster.cu)
constexpr uint64_t OPEN_NONE = 0, OPEN_UNKNOWN = 1, OPEN_BIAS = 2;
constexpr int NO_POS = 0x7fffffff;

struct ScanShared {
    uint64_t full_bar[SC_STAGES];
    uint64_t x_in;                // open-cluster state entering the tile            (warp 0, between the barriers (A) and (B))
    uint32_t prefix;              // segment index of the record of the tile's kept END of rank 0 (one less when the carried END is not written)
    uint32_t adj;                 // bit 0: the carried END is not written by this tile; bit 1: it is the chunk's head
    uint32_t open_after[2];       // (interior tiles) a cluster is open after the tile's last position; by tile parity (read after (B))
    uint32_t wsum[SC_WARPS];      // per warp: #kept ENDs | #ENDs << 16
    uint32_t bS[2][SC_WARPS];     // per warp: lanes whose START word is not empty (by tile parity, like sS)
    int wfe[SC_WARPS];            // first END of the warp (tile-local position), NO_POS = none
    int wle[2][SC_WARPS];         // last END of the warp, -1 = none (tiles at the edges of the shard only); by tile parity
    unsigned int hist[E2S_HIST_BINS];
    uint64_t sS[2][SC_THREADS];   // START words of the tile, by tile parity: read until the tile's records are out
    uint16_t e_ent[SC_CAP];       // tile-local positions of the kept ENDs, by rank
    // chunk state that lives here instead of in (every thread's) registers: the kernel runs at its 64-register cap
    uint64_t x_state;             // warp 0: open-cluster state after the last tile; unknown until the chunk's first event
    uint64_t n_end_acc;           // warp 0: ENDs seen (head included)
    uint64_t head_end;            // warp 0: 1 + global position of the chunk's head END, 0 = none
    unsigned long long big_bases; // sum of the written lengths above MAX_C_LEN (the others are in hist)
    uint32_t seen;                // warp 0: the chunk has had an event
};

__device__ __forceinline__ void tma_load_2d_u8(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void bulk_g2s_a(uint32_t dst, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// loads from the stages by 32-bit shared-window address (volatile: the data is written by the copy engine between two
// visits of the same address)
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint2 lds_u64(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds_u128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u64(uint32_t addr, uint32_t lo, uint32_t hi) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(lo), "r"(hi) : "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ uint64_t shfl64(uint64_t v, int src) {
    return (uint64_t(__shfl_sync(FULL, uint32_t(v >> 32), src)) << 32) | __shfl_sync(FULL, uint32_t(v), src);
}
// one step of the bit-sliced "value < k" from the least significant plane up: lt' = k_b ? (~x | lt) : (~x & lt), with
// km = all ones / zero for k_b -- one 3-input logic function (LOP3, table 0x8E), km read from the kernel parameters
__device__ __forceinline__ uint32_t lt_step(uint32_t x, uint32_t km, uint32_t lt) {
    uint32_t r;  // (written as C++ the compiler emits three instructions for it)
    asm("lop3.b32 %0, %1, %2, %3, 0x8E;" : "=r"(r) : "r"(x), "r"(km), "r"(lt));
    return r;
}
// nearest set bit at or before tile-local position e of a 16 384-bit mask kept as one 64-bit word per thread (at the
// shared-window address words) plus, per warp, the ballot of the lanes whose word is not empty (at bal) and the warps that
// have any (any8); -1 = none
__device__ __forceinline__ int find_prev(uint32_t words, uint32_t bal, uint32_t any8, uint32_t e) {
    uint32_t t = e >> 6;
    uint2 v = lds_u64(words + t * 8u);
    const uint32_t keep = FULL >> (31u - (e & 31u));
    if (e & 32u) v.y &= keep;
    else {
        v.x &= keep;
        v.y = 0;
    }
    if (!(v.x | v.y)) {
        uint32_t w = t >> 5;
        uint32_t bm = lds_u32(bal + w * 4u) & ((1u << (t & 31u)) - 1u);
        if (!bm) {
            const uint32_t a8 = any8 & ((1u << w) - 1u);
            if (!a8) return -1;
            w = 31u - uint32_t(__clz(a8));
            bm = lds_u32(bal + w * 4u);
        }
        t = w * 32u + 31u - uint32_t(__clz(bm));
        v = lds_u64(words + t * 8u);
    }
    return int(t * 64u) + (v.y ? 63 - __clz(v.y) : 31 - __clz(v.x));
}

}  // namespace

// OCC = the resident CTAs per SM ptxas is asked to make room for.  Its register allocation is erratic around the 64-register
// line (the same source has come out at 56 / 62 registers for OCC = 4 and 62 / 72 / 80 for OCC = 3, and the 56-register
// build re-materialises per-thread constants every tile: C2 253.5 vs 247.7 us), so both builds are compiled and
// scan_kernel() picks at run time: most resident CTAs first, then most registers.
template <int OCC>
__global__ void __launch_bounds__(SC_THREADS, OCC) k_cluster_scan(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ Scan8Params p) {
    extern __shared__ __align__(128) uint8_t smem_dyn[];  // SC_STAGES stages, then SC_PSLOTS plane windows
    __shared__ ScanShared sh;
    const uint32_t stage0 = smem_u32(smem_dyn);
    const uint32_t planes0 = stage0 + SC_STAGES * SC_STAGE_BYTES;
    const uint32_t sS0 = smem_u32(&sh.sS[0][0]), bS0 = smem_u32(&sh.bS[0][0]);  // shared-window addresses of the double-buffered arrays

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool pf = p.pf_mcov != 0;
    const int spread = p.min_len >= 2 ? p.min_len - 2 : -1;  // extra positions a START shadows; -1: nothing is dropped
    const uint32_t c = blockIdx.x;
    const uint32_t t_lo = c * p.tiles_per_chunk < p.num_tiles ? c * p.tiles_per_chunk : p.num_tiles;
    const uint32_t t_hi = t_lo + p.tiles_per_chunk < p.num_tiles ? t_lo + p.tiles_per_chunk : p.num_tiles;
    const uint32_t n_my = t_hi - t_lo;
    uint64_t* const seg_start = p.seg_start + uint64_t(c) * p.seg_cap;  // my chunk's segment
    uint16_t* const seg_len = p.seg_len + uint64_t(c) * p.seg_cap;
    const uint32_t seg_room = uint32_t(p.seg_cap < 0xffffffffull ? p.seg_cap : 0xffffffffull);

    // where my words are in a stage: run b of my warp's block at own + 256 b; the word before it in the same run (lane 0:
    // the last word of the previous block) and the word after it, at the same constant offsets from their bases.  Thread 0
    // and the last thread read next to the stage there and take their neighbours from the edge boxes afterwards.
    const uint32_t own = uint32_t(warp) * LCPT_BLOCK + uint32_t(lane) * 8u;
    const uint32_t prev_off = own + (lane ? 0u - 8u : 0u - 1800u) + 4u;  // high half: bit 63
    const uint32_t next_off = own + (lane < 31 ? 8u : 1800u);            // low half: bit 0

    for (int i = tid; i < E2S_HIST_BINS; i += SC_THREADS) sh.hist[i] = 0;
    auto issue = [&](uint32_t it) {  // thread 0: the it-th tile of the chunk -> stage it % SC_STAGES
        if (it >= n_my) return;
        const int stage = int(it % SC_STAGES);
        const uint32_t dst = stage0 + uint32_t(stage) * SC_STAGE_BYTES;
        const uint32_t t = t_lo + it;
        mbar_expect_tx(&sh.full_bar[stage], SC_STAGE_BYTES + (pf ? SC_PF_BYTES : 0));
        // (block 0 of the array = the LCPT_BLOCK positions before local position 0: tile t = blocks 8 t + 1 .. 8 t + 8)
        bulk_g2s_a(dst + SC_EDGE, p.lcpt + (uint64_t(t) * SC_WARPS + 1) * LCPT_BLOCK, SC_T, &sh.full_bar[stage]);
        // the tensor: rows of 256 bytes = one run; words 30, 31 of the 8 runs of the block before, words 0, 1 of the block after
        tma_load_2d_u8(dst, &tmap, 240, int(t * SC_WARPS * 8), &sh.full_bar[stage]);
        tma_load_2d_u8(dst + SC_EDGE + SC_T, &tmap, 0, int((t * SC_WARPS + SC_WARPS + 1) * 8), &sh.full_bar[stage]);
        if (pf) bulk_g2s_a(planes0 + (it % SC_PSLOTS) * SC_PF_STRIDE, p.planes + uint64_t(t) * (SC_T / 64), SC_PF_BYTES, &sh.full_bar[stage]);
    };
    if (tid == 0) {
        sh.x_state = OPEN_UNKNOWN;
        sh.n_end_acc = 0;
        sh.head_end = 0;
        sh.big_bases = 0;
        sh.seen = 0;
        for (int s = 0; s < SC_STAGES; ++s) mbar_init(&sh.full_bar[s], 1);
        fence_mbar_init();
        for (uint32_t s = 0; s < uint32_t(SC_STAGES); ++s) issue(s);
    }
    __syncthreads();

    // chunk state (warp 0; identical in its lanes); the rest of it is in shared memory (ScanShared)
    uint32_t cnt = 0;            // records written to the segment so far (a segment holds fewer than 2^32)

    uint32_t pf_win = planes0;  // the tile's plane window: slot it % SC_PSLOTS
    for (uint32_t it = 0; it < n_my; ++it, pf_win = pf_win == planes0 + (SC_PSLOTS - 1) * SC_PF_STRIDE ? planes0 : pf_win + SC_PF_STRIDE) {
        const uint32_t pb = it & 1u;  // = stage (SC_STAGES == 2)
        const uint32_t parity = (it >> 1) & 1u;
        const uint32_t t = t_lo + it;
        const uint32_t sa = stage0 + pb * SC_STAGE_BYTES + SC_EDGE;  // the tile's first byte; the edge boxes at sa - SC_EDGE and sa + SC_T
        const bool interior = t >= p.t_int_lo && t < p.t_int_hi;
        const uint32_t sS_a = sS0 + pb * (SC_THREADS * 8u), bS_a = bS0 + pb * (SC_WARPS * 4u);
        const int stage = int(pb);

        mbar_wait(&sh.full_bar[stage], parity);

        // ---- G = (lcp >= k) and A of my 64 positions; G and A of the position before and of the position after them
        uint64_t G, A;
        uint32_t g_m1, a_m1, g_p, a_p;  // bit 0: position -1 / position 64 of my word
        {
            uint32_t lt_lo = 0, lt_hi = 0, ltp = 0, ltn = 0;
#pragma unroll
            for (int b = 0; b < 7; ++b) {
                const uint2 v = lds_u64(sa + own + 256u * b);
                lt_lo = lt_step(v.x, p.km[b], lt_lo);
                lt_hi = lt_step(v.y, p.km[b], lt_hi);
                ltp = lt_step(lds_u32(sa + prev_off + 256u * b), p.km[b], ltp);
                ltn = lt_step(lds_u32(sa + next_off + 256u * b), p.km[b], ltn);
            }
            const uint2 av = lds_u64(sa + own + 256u * 7);
            uint32_t ap = lds_u32(sa + prev_off + 256u * 7), an = lds_u32(sa + next_off + 256u * 7);
            if (tid == 0) {  // the group before the tile: word 31 of the runs of the block before it (edge box: rows of {word 30, word 31})
                ltp = 0;
#pragma unroll
                for (int b = 0; b < 7; ++b) ltp = lt_step(lds_u32(sa - SC_EDGE + 12u + 16u * b), p.km[b], ltp);
                ap = lds_u32(sa - SC_EDGE + 12u + 16u * 7);
            }
            if (tid == SC_THREADS - 1) {  // the group after the tile: word 0 of the runs of the block after it
                ltn = 0;
#pragma unroll
                for (int b = 0; b < 7; ++b) ltn = lt_step(lds_u32(sa + SC_T + 16u * b), p.km[b], ltn);
                an = lds_u32(sa + SC_T + 16u * 7);
            }
            G = ~((uint64_t(lt_hi | p.km[7]) << 32) | (lt_lo | p.km[7]));  // km[7]: "every value is below k" (k >= 128)
            A = (uint64_t(av.y) << 32) | av.x;
            g_m1 = (~(ltp | p.km[7])) >> 31;
            a_m1 = ap >> 31;
            g_p = (~(ltn | p.km[7])) & 1u;
            a_p = an & 1u;
        }

        // ---- START / END masks of my 64 positions
        uint64_t S, E;
        {
            const uint64_t Gn = (G >> 1) | (uint64_t(g_p) << (SC_V - 1));  // ge(j+1)
            const uint64_t An = (A >> 1) | (uint64_t(a_p) << (SC_V - 1));  // lcp[j] > lcp[j+1]
            E = G & ((A & ~An) | ~Gn);
            // END of the position before mine: ge(-1) & ((A(-1) & ~A(0)) | ~ge(0))
            uint64_t e_prev = uint64_t(g_m1 & ((a_m1 & ~uint32_t(A)) | ~uint32_t(G)) & 1u);
            uint64_t vm = ~uint64_t(0);
            if (!interior) {  // first tile of the eBWT, the tile holding position n_global - 1, tiles reaching past n_local
                const uint64_t my_base = uint64_t(t) * SC_T + uint64_t(tid) * SC_V;
                const uint64_t gpos = p.global_off + my_base;
                if (gpos == 0) {  // the init special cases of ref:ebwt2clust.cpp:83-86
                    E &= ~uint64_t(1);
                    e_prev = 0;
                    if ((G & 1u) && !(G & 2u)) E |= 2u;
                }
                const int64_t nvalid = int64_t(p.n_local) - int64_t(my_base);
                vm = nvalid >= SC_V ? ~uint64_t(0) : (nvalid <= 0 ? 0 : ((uint64_t(1) << nvalid) - 1));
                const int64_t last = int64_t(p.n_global) - 1 - int64_t(gpos);  // END(n_global-1): host tail rule
                if (last >= 0 && last < SC_V) E &= ~(uint64_t(1) << last);
                E &= vm;
            }
            const uint64_t Gp = (G << 1) | g_m1;
            const uint64_t Ep = (E << 1) | e_prev;
            S = G & (~Gp | Ep) & vm;
        }
        sts_u64(sS_a + uint32_t(tid) * 8u, uint32_t(S), uint32_t(S >> 32));

        // ---- K = kept ENDs: E minus the ENDs of clusters shorter than min_len (a START at the same position or up to `spread`
        // positions before).  Before the tile: no START assumed -- the one END that can pair with a START of an earlier tile
        // is the tile's first event, which warp 0 tests exactly below.
        uint64_t K = E;
        if (spread >= 0) {
            uint64_t sm = S;
            if (spread >= 1) {  // (kernel-uniform) the previous thread's START word
                __syncthreads();
                uint64_t lo = tid ? sh.sS[pb][tid - 1] : 0;
                uint64_t hi = S;
                int width = 1;  // sm = OR of (S << d), d = 0 .. width - 1, over the 128 bits lo:hi
                while (2 * width <= spread + 1) {
                    hi |= (hi << width) | (lo >> (64 - width));
                    lo |= lo << width;
                    width *= 2;
                }
                const int rest = spread + 1 - width;
                if (rest) hi |= (hi << rest) | (lo >> (64 - rest));
                sm = hi;
            }
            K = E & ~sm;
        }
        uint32_t k_lo = uint32_t(K), k_hi = uint32_t(K >> 32);

        // ---- ranks of the kept ENDs (one block scan of #kept | #ENDs << 16) and the per-warp summaries
        const uint32_t pk = uint32_t(__popc(k_lo) + __popc(k_hi)) | (uint32_t(__popcll(E)) << 16);
        uint32_t inc = pk;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(FULL, inc, d);
            if (lane >= d) inc += o;
        }
        {
            const uint32_t bS = __ballot_sync(FULL, S != 0), bE = __ballot_sync(FULL, E != 0);
            int fe = NO_POS;
            if (bE) {  // (warp-uniform) the warp's first END: in the word of the first lane that has one
                const int src = __ffs(bE) - 1;
                const uint32_t e_lo = __shfl_sync(FULL, uint32_t(E), src), e_hi = __shfl_sync(FULL, uint32_t(E >> 32), src);
                fe = (warp * 32 + src) * SC_V + (e_lo ? __ffs(e_lo) - 1 : 31 + __ffs(e_hi));
            }
            if (lane == 31) sh.wsum[warp] = inc;
            if (lane == 0) {
                sts_u32(bS_a + uint32_t(warp) * 4u, bS);
                sh.wfe[warp] = fe;
            }
            if (interior) {  // a cluster is open after the tile iff its last position is inside one and not its END
                if (tid == SC_THREADS - 1) sh.open_after[pb] = uint32_t((G & ~E) >> 63);
            } else {         // (positions past n_local, the cleared END(n_global - 1): by the tile's last START / END)
                int le = -1;
                if (bE) {
                    const int src = 31 - __clz(bE);
                    const uint64_t El = shfl64(E, src);
                    le = (warp * 32 + src) * SC_V + 63 - __clzll(El);
                }
                if (lane == 0) sh.wle[pb][warp] = le;
            }
        }
        __syncthreads();  // (A) per-warp summaries, START words.  Every thread has this tile's words in registers: the stage is refilled
        if (tid == 0) issue(it + SC_STAGES);

        // my warp's rank offset, the tile's totals, the warps that have a START
        uint32_t baseK, nK, nE, any8;
        {
            const uint32_t ws = sh.wsum[lane & (SC_WARPS - 1)], bq = lds_u32(bS_a + uint32_t(lane & (SC_WARPS - 1)) * 4u);
            const uint32_t tot = __reduce_add_sync(FULL, lane < SC_WARPS ? ws : 0u);
            const uint32_t base = (inc - pk) + __reduce_add_sync(FULL, lane < warp ? ws : 0u);
            any8 = __ballot_sync(FULL, bq != 0) & ((1u << SC_WARPS) - 1u);
            nK = tot & 0xffffu;
            nE = tot >> 16;
            baseK = base & 0xffffu;
        }

        // ---- warp 0, before the barrier (B): the carried END and where the tile's records go
        int t_fe = NO_POS;
        if (warp == 0) {
            const uint64_t tile_gbase = p.global_off + uint64_t(t) * SC_T;
            int t_fs = NO_POS;
            if (any8) {
                const uint32_t w = uint32_t(__ffs(any8) - 1);
                const uint32_t t2 = w * 32u + uint32_t(__ffs(lds_u32(bS_a + w * 4u)) - 1);
                const uint2 v = lds_u64(sS_a + t2 * 8u);
                t_fs = int(t2 * 64u) + (v.x ? __ffs(v.x) - 1 : 31 + __ffs(v.y));
            }
#pragma unroll
            for (int q = SC_WARPS - 1; q >= 0; --q)
                if (sh.wfe[q] != NO_POS) t_fe = sh.wfe[q];
            // the tile's first event is an END: its START lies before the tile (a START and an END at the same position: the
            // START comes first, t_fe == t_fs is not carried)
            const bool carried = t_fe != NO_POS && t_fe < t_fs;
            // The carried END is tested exactly on the wrapped length (ref:ebwt2clust.cpp:56,104) against the carried-in START: it is
            // the only END of the tile that can be 65 536 or more positions from its START.  Before the chunk's first event that
            // START is not known here: the END is the chunk's head, left to k_chunk_resolve.
            uint32_t adj = 0;  // 1: the carried END is not written by this tile
            const uint64_t X = sh.x_state;
            const bool seen = sh.seen != 0;
            const bool is_head = carried && !seen;
            if (carried) {
                adj = 1;
                if (seen && X >= OPEN_BIAS) {
                    const uint32_t len = uint32_t(tile_gbase + uint64_t(t_fe) - (X - OPEN_BIAS) + 1) & 0xffffu;
                    adj = int(len) >= p.min_len ? 0u : 1u;
                }
                if (is_head && lane == 0) sh.head_end = tile_gbase + uint64_t(t_fe) + 1;
            }
            if (lane == 0) {
                sh.n_end_acc += nE;
                sh.x_in = X;
                sh.prefix = cnt - ((carried && adj) ? 1u : 0u);  // (the records after a carried END that is not written move up one)
                sh.adj = adj | (is_head ? 2u : 0u);
            }
            cnt += nK - adj;
        }

        // ---- scatter: the tile-local positions of my kept ENDs to their ranks (the list window by window of SC_CAP: one
        // iteration unless the tile is unusually dense)
        for (uint32_t win = 0; win == 0 || win < nK; win += SC_CAP) {
            if (win) __syncthreads();  // the previous window's list is no longer read
            {
                uint32_t r = baseK - win;  // (mod 2^32: ranks below the window fail the bound check)
                uint32_t mlo = k_lo, mhi = k_hi;
                const uint32_t p0 = uint32_t(tid) * SC_V;
                if (nK <= uint32_t(SC_CAP)) {  // (the usual case: every rank is inside the window)
                    while (mlo | mhi) {
                        const uint32_t x = mlo ? mlo : mhi;
                        const uint32_t b = uint32_t(__ffs(x) - 1) + (mlo ? 0u : 32u);
                        if (mlo) mlo &= mlo - 1;
                        else mhi &= mhi - 1;
                        sh.e_ent[r++] = uint16_t(p0 + b);
                    }
                } else {
                    while (mlo | mhi) {
                        const uint32_t x = mlo ? mlo : mhi;
                        const uint32_t b = uint32_t(__ffs(x) - 1) + (mlo ? 0u : 32u);
                        if (mlo) mlo &= mlo - 1;
                        else mhi &= mhi - 1;
                        if (r < uint32_t(SC_CAP)) sh.e_ent[r] = uint16_t(p0 + b);
                        ++r;
                    }
                }
            }
            __syncthreads();  // (B) list; warp 0's tile words; warp 0 is done with the summaries

            // ---- the tile that holds position n_global - 2 (one per eBWT): an END there decides the reference's post-EOF phantom
            // value (SURVEY.md A3) whether its record is kept or not
            if (!interior && win == 0) {
                const uint64_t tile_gbase = p.global_off + uint64_t(t) * SC_T;
                if (p.n_global - 2 - tile_gbase < uint64_t(SC_T)) {
                    const uint32_t e_loc = uint32_t(p.n_global - 2 - tile_gbase);
                    if (uint32_t(tid) == (e_loc >> 6) && ((E >> (e_loc & 63)) & 1u)) {
                        const int s_loc = find_prev(sS_a, bS_a, any8, e_loc);
                        if (s_loc >= 0) p.res->end_nm2_start = tile_gbase + uint64_t(s_loc) + 1;
                        else if (!(sh.adj & 2u)) p.res->end_nm2_start = sh.x_in >= OPEN_BIAS ? sh.x_in - OPEN_BIAS + 1 : ~0ull;
                        // (the chunk's head: k_chunk_resolve answers)
                    }
                }
            }
            if (warp == 0 && win == 0) {  // the chunk state after this tile (off the other warps' path to the records)
                const int t_ls = find_prev(sS_a, bS_a, any8, SC_T - 1);
                bool open_after;
                if (interior) {
                    open_after = sh.open_after[pb] != 0;
                } else {
                    int t_le = -1;
#pragma unroll
                    for (int q = 0; q < SC_WARPS; ++q)
                        if (sh.wle[pb][q] >= 0) t_le = sh.wle[pb][q];
                    open_after = t_ls > t_le;
                }
                if ((t_ls >= 0 || t_fe != NO_POS) && lane == 0) {  // (read again by warp 0 after the next tile's barrier (A))
                    const uint64_t tile_gbase = p.global_off + uint64_t(t) * SC_T;
                    sh.x_state = (open_after && t_ls >= 0) ? tile_gbase + uint64_t(t_ls) + OPEN_BIAS : (open_after ? sh.x_in : OPEN_NONE);
                    sh.seen = 1;
                }
            }
            if (nK == 0) break;

            const uint32_t prefix = sh.prefix + win;
            const uint32_t n_win = nK - win < uint32_t(SC_CAP) ? nK - win : uint32_t(SC_CAP);
            // entry -> lane: the first SC_THREADS entries in order, later rounds from the last thread down (warp 0 carries the chunk
            // state: the extra rounds land on the warps that are ahead)
            for (uint32_t i = uint32_t(tid), nxt = 2u * SC_THREADS - 1u - uint32_t(tid); i < n_win; i = nxt, nxt += SC_THREADS) {
                const uint32_t e = sh.e_ent[i];
                const int s_loc = find_prev(sS_a, bS_a, any8, e);
                uint32_t len, o = prefix + i;
                uint32_t b_lo;          // first position of the analysed range, from the plane window's first position (tile start - PL_PAD)
                bool in_window = true;  // ... unless the range starts before it (a wrapped length)
                uint64_t st;
                if (s_loc >= 0) {
                    len = e - uint32_t(s_loc) + 1u;
                    b_lo = uint32_t(s_loc) + PL_PAD;
                    st = (p.global_off + uint64_t(t) * SC_T) + uint32_t(s_loc);
                } else {  // no START in the tile before it: the tile's carried END (rank 0)
                    if (sh.adj) continue;  // the chunk's head (k_chunk_resolve writes it) / dropped by the exact test
                    const uint64_t tile_gbase = p.global_off + uint64_t(t) * SC_T;
                    st = sh.x_in - OPEN_BIAS;
                    len = uint32_t(tile_gbase + e - st + 1) & 0xffffu;
                    in_window = st + PL_PAD >= tile_gbase;
                    b_lo = uint32_t(st + PL_PAD - tile_gbase);
                }
                if (o < seg_room) {
                    seg_start[o] = st;
                    seg_len[o] = uint16_t(len);
                } else {
                    p.res->overflow |= 1;
                }
                if (len <= uint32_t(MAX_C_LEN)) atomicAdd(&sh.hist[len], 1u);
                else atomicAdd(&sh.big_bases, (unsigned long long)len);
                // BWT prefilter: the one-popcount bound (planes.cuh) on the analysed range [st, st + len) in the plane window, one
                // quad {plane 0 lo, hi, plane 1 lo, hi} = 64 positions per step; a record whose range starts before the window goes
                // straight to the exact test
                if (pf && len >= 2 * p.pf_mcov && len <= uint32_t(MAX_C_LEN)) {
                    bool pass = true;
                    if (in_window) {
                        const uint32_t b_last = b_lo + len - 1;
                        uint32_t q = b_lo >> 6;
                        const uint32_t q_last = b_last >> 6;
                        uint32_t addr = pf_win + q * 16u;
                        uint4 pv = lds_u128(addr);  // {plane 0 lo, hi, plane 1 lo, hi} of 64 positions
                        const uint32_t s5 = b_lo & 31u;
                        const bool s_hi = (b_lo & 32u) != 0;
                        const uint32_t f0 = 0u - (((s_hi ? pv.y : pv.x) >> s5) & 1u), f1 = 0u - (((s_hi ? pv.w : pv.z) >> s5) & 1u);  // the first record's code
                        uint32_t mlo = s_hi ? 0u : FULL << s5, mhi = s_hi ? FULL << s5 : FULL;
                        uint32_t others = 0;
                        while (q < q_last) {
                            others += __popc(((pv.x ^ f0) | (pv.z ^ f1)) & mlo) + __popc(((pv.y ^ f0) | (pv.w ^ f1)) & mhi);
                            ++q;
                            addr += 16u;
                            pv = lds_u128(addr);
                            mlo = mhi = FULL;
                        }
                        const uint32_t e5 = 31u - (b_last & 31u);
                        const bool e_hi = (b_last & 32u) != 0;
                        mlo &= e_hi ? FULL : FULL >> e5;
                        mhi &= e_hi ? FULL >> e5 : 0u;
                        others += __popc(((pv.x ^ f0) | (pv.z ^ f1)) & mlo) + __popc(((pv.y ^ f0) | (pv.w ^ f1)) & mhi);
                        pass = others >= p.pf_mcov;  // at least mcov records differ from the first one's base code
                    }
                    if (pass) {
                        const unsigned long long at = atomicAdd(&p.res->n_pf, 1ull);
                        if (at < p.pf_cap) p.pf_list[at] = SurvEntry{st, st - p.global_off, len, 0u};
                        else p.res->overflow |= 2;  // (seen by every rank in the exchange rows: all of them repeat the round)
                    }
                }
            }
        }
    }

    // ---- what the chunk leaves for k_chunk_resolve
    __syncthreads();
    unsigned long long acc_bases = tid == 0 ? sh.big_bases : 0ull;  // sum of the written lengths: from the histogram
    for (int i = tid; i < E2S_HIST_BINS; i += SC_THREADS)
        if (sh.hist[i]) {
            atomicAdd(&p.res->hist[i], (unsigned long long)sh.hist[i]);
            acc_bases += (unsigned long long)sh.hist[i] * uint32_t(i);
        }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc_bases += __shfl_xor_sync(FULL, acc_bases, d);
    ChunkRec* cr = p.chunks + c;
    if (lane == 0 && acc_bases) atomicAdd(&cr->n_bases, acc_bases);
    if (tid == 0) {
        const uint64_t X = sh.x_state;
        cr->own_count = cnt;
        cr->head_end = sh.head_end;
        cr->last_state = sh.seen ? (X >= OPEN_BIAS ? X : 1ull) : 0ull;  // 0: no event; 1: closed; >= 2: OPEN_BIAS + global START
        cr->n_end = sh.n_end_acc;
        // the chunk's last record (written by some thread of this CTA before the barrier above)
        if (cnt && cnt - 1 < seg_room) cr->last_len = seg_len[cnt - 1];
        if (c == 0 && p.tail_lcp) {
            p.res->tail_lcp_nm2 = p.tail_lcp[0];
            p.res->tail_lcp_nm1 = p.tail_lcp[1];
            p.res->tail_bwt_nm1 = p.tail_bwt[0];
        }
    }
}

// =============================================================================================
// k_chunk_resolve: what the chunks could not know (one CTA; a few hundred chunks)
// =============================================================================================
// state entering a chunk = state left by the nearest earlier chunk that had an event (else the state before the shard);
// the chunk's head END closes the cluster that state holds open: exact length test, one record in front of the chunk's own;
// an END without any START in the shard is the SHARD's head (resolved by e2s_cluster_merge across shards).  Then the
// exclusive scan of the chunks' record counts (= where each segment goes in the position-ordered list) and the shard totals.
constexpr int RS_THREADS = 1024;

__global__ void __launch_bounds__(RS_THREADS) k_chunk_resolve(ResolveParams p) {
    __shared__ unsigned long long s_state[RS_THREADS];
    __shared__ unsigned long long s_cnt[RS_THREADS];
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_tot[4];  // records, ENDs, bases, (last chunk with records) + 1
    const int c = threadIdx.x, lane = c & 31, warp = c >> 5;
    const bool act = uint32_t(c) < p.n_chunks;
    ChunkRec rec;
    rec.own_count = rec.head_end = rec.last_state = rec.n_end = rec.n_bases = rec.last_len = 0;
    if (act) rec = p.chunks[c];
    s_state[c] = rec.last_state;
    if (c < 4) s_tot[c] = 0;
    __syncthreads();
    uint64_t X = p.init_state;
    if (act && rec.head_end)  // (only a head END asks what was open before the chunk; the threads past the last chunk would walk all the way down)
        for (int j = c - 1; j >= 0; --j)
            if (s_state[j]) {
                X = s_state[j] >= OPEN_BIAS ? s_state[j] : OPEN_NONE;
                break;
            }
    uint64_t h_start = 0;
    uint32_t h_len = 0, h_kept = 0;
    if (act && rec.head_end) {
        const uint64_t e = rec.head_end - 1;
        if (X >= OPEN_BIAS) {
            h_start = X - OPEN_BIAS;
            h_len = uint32_t(e - h_start + 1) & 0xffffu;  // append_entry's wrapped length (ref:ebwt2clust.cpp:56,104)
            h_kept = int(h_len) >= p.min_len ? 1u : 0u;
            if (e + 2 == p.n_global) p.res->end_nm2_start = h_start + 1;
        } else {  // no START in this shard: the shard's head
            p.res->head_end = e + 1;
            if (e + 2 == p.n_global) p.res->end_nm2_start = ~0ull;
        }
    }
    const unsigned long long mine = rec.own_count + h_kept;
    unsigned long long inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = shfl64(inc, lane >= d ? lane - d : lane);
        if (lane >= d) inc += o;
    }
    if (lane == 31) s_warp[warp] = inc;
    s_cnt[c] = mine;
    __syncthreads();
    unsigned long long off = inc - mine;
    for (int q = 0; q < warp; ++q) off += s_warp[q];
    if (act) {
        ChunkSeg sg;
        sg.off = off;
        sg.own_count = rec.own_count;
        sg.head_start = h_start;
        sg.head_len = h_len;
        sg.head_kept = h_kept;
        p.segs[c] = sg;
        if (h_kept) {
            if (h_len <= uint32_t(MAX_C_LEN)) atomicAdd(&p.res->hist[h_len], 1ull);
            // the head record's turn at the fused BWT prefilter (its positions lie before the chunk: global planes)
            if (p.pf_mcov && h_len >= 2 * p.pf_mcov && h_len <= uint32_t(MAX_C_LEN)) {
                bool pass = h_start < p.global_off;  // (cannot happen for a record with a known START; kept for safety)
                if (!pass) pass = frequent_bound(p.planes, int64_t(h_start - p.global_off), h_len, p.pf_mcov);
                if (pass) {
                    const unsigned long long at = atomicAdd(&p.res->n_pf, 1ull);
                    if (at < p.pf_cap) p.pf_list[at] = SurvEntry{h_start, h_start - p.global_off, h_len, 0u};
                    else p.res->overflow |= 2;
                }
            }
        }
    }
    {   // block totals: warp sums by shuffles, one shared atomic per warp
        unsigned long long w0 = act ? mine : 0, w1 = act ? rec.n_end : 0, w2 = act ? rec.n_bases + (h_kept ? h_len : 0u) : 0;
        unsigned long long w3 = (act && mine) ? (unsigned long long)(c + 1) : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            w0 += shfl64(w0, lane ^ d);
            w1 += shfl64(w1, lane ^ d);
            w2 += shfl64(w2, lane ^ d);
            const unsigned long long o = shfl64(w3, lane ^ d);
            w3 = o > w3 ? o : w3;
        }
        if (lane == 0) {
            if (w0) atomicAdd(&s_tot[0], w0);
            if (w1) atomicAdd(&s_tot[1], w1);
            if (w2) atomicAdd(&s_tot[2], w2);
            if (w3) atomicMax(&s_tot[3], w3);
        }
    }
    __syncthreads();
    if (act && mine && s_tot[3] == (unsigned long long)(c + 1))  // the list's last record is this chunk's last
        p.res->last_rec = (s_tot[0] << 16) | (rec.own_count ? rec.last_len : h_len);
    if (c == 0) {
        p.res->n_written = s_tot[0];
        p.res->n_end = s_tot[1];
        p.res->n_bases = s_tot[2];
        uint64_t x_out = p.init_state;
        bool any = false;
        for (int j = int(p.n_chunks) - 1; j >= 0; --j)
            if (s_state[j]) {
                x_out = s_state[j] >= OPEN_BIAS ? s_state[j] : OPEN_NONE;
                any = true;
                break;
            }
        p.res->any_event = any ? 1ull : 0ull;
        p.res->open_start = x_out >= OPEN_BIAS ? x_out - OPEN_BIAS + 1 : 0;
    }
}

// segments -> position-ordered contiguous list: as SoA (start u64, len u16) or as the 10-byte records of the .clusters
// file (ref:ebwt2clust.cpp:58-59)
__global__ void __launch_bounds__(256) k_export_records(const ChunkSeg* __restrict__ segs, uint32_t n_chunks, uint64_t seg_cap,
                                                        const uint64_t* __restrict__ seg_start, const uint16_t* __restrict__ seg_len,
                                                        uint64_t* __restrict__ out_start, uint16_t* __restrict__ out_len,
                                                        uint16_t* __restrict__ out_packed) {
    for (uint32_t c = blockIdx.y; c < n_chunks; c += gridDim.y) {
        const ChunkSeg sg = segs[c];
        const uint64_t total = sg.own_count + sg.head_kept;
        const uint64_t src0 = uint64_t(c) * seg_cap;
        for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += uint64_t(gridDim.x) * blockDim.x) {
            uint64_t st;
            uint16_t ln;
            if (sg.head_kept && i == 0) {
                st = sg.head_start;
                ln = uint16_t(sg.head_len);
            } else {
                st = seg_start[src0 + i - sg.head_kept];
                ln = seg_len[src0 + i - sg.head_kept];
            }
            const uint64_t o = sg.off + i;
            if (out_packed) {
                uint16_t* q = out_packed + o * 5;
                q[0] = uint16_t(st);
                q[1] = uint16_t(st >> 16);
                q[2] = uint16_t(st >> 32);
                q[3] = uint16_t(st >> 48);
                q[4] = ln;
            } else {
                out_start[o] = st;
                out_len[o] = ln;
            }
        }
    }
}

// =============================================================================================
// host side
// =============================================================================================
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled scan_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    }
    return fn;
}

uint64_t scan_num_tiles(uint64_t n_local) { return (n_local + SC_T - 1) / SC_T; }

using ScanKernel = void (*)(const CUtensorMap, const Scan8Params);
// the build that keeps the most CTAs resident, among equals the one ptxas gave more registers (E2S_SCAN_OCC=3|4 forces one)
static ScanKernel scan_kernel() {
    static const ScanKernel chosen = [] {
        const ScanKernel k3 = static_cast<ScanKernel>(k_cluster_scan<3>), k4 = static_cast<ScanKernel>(k_cluster_scan<SC_OCC>);
        if (const char* e = getenv("E2S_SCAN_OCC")) {
            if (atoi(e) == 3) return k3;
            if (atoi(e) == SC_OCC) return k4;
        }
        int o3 = 0, o4 = 0;
        cudaFuncAttributes a3{}, a4{};
        cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, int(SC_DYN_SMEM));
        cudaFuncSetAttribute(k4, cudaFuncAttributeMaxDynamicSharedMemorySize, int(SC_DYN_SMEM));
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o3, k3, SC_THREADS, SC_DYN_SMEM) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o4, k4, SC_THREADS, SC_DYN_SMEM) != cudaSuccess ||
            cudaFuncGetAttributes(&a3, k3) != cudaSuccess || cudaFuncGetAttributes(&a4, k4) != cudaSuccess) {
            cudaGetLastError();
            return k4;
        }
        return (o3 > o4 || (o3 == o4 && a3.numRegs > a4.numRegs)) ? k3 : k4;
    }();
    return chosen;
}

static int scan_occupancy(int* out) {
    static int occ_dev[64] = {0};  // function attributes are per device
    int dev = 0;
    cudaGetDevice(&dev);
    int& occ = occ_dev[dev & 63];
    if (!occ) {
        cudaError_t e = cudaFuncSetAttribute(scan_kernel(), cudaFuncAttributeMaxDynamicSharedMemorySize, int(SC_DYN_SMEM));
        if (e != cudaSuccess) return int(e);
        int o = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, scan_kernel(), SC_THREADS, SC_DYN_SMEM);
        if (e != cudaSuccess) return int(e);
        if (o < 1) return int(cudaErrorLaunchOutOfResources);
        occ = o;
    }
    *out = occ;
    return 0;
}

// chunks of a shard: one per CTA the device holds at once (at most SCAN_MAX_CHUNKS), at least one tile each
cudaError_t scan_plan(uint64_t n_local, int sm_count, uint32_t* n_chunks, uint32_t* tiles_per_chunk) {
    int occ = 0;
    const int rc = scan_occupancy(&occ);
    if (rc) return cudaError_t(rc);
    const uint64_t nt = scan_num_tiles(n_local);
    uint64_t g = uint64_t(sm_count) * occ;
    if (g > SCAN_MAX_CHUNKS) g = SCAN_MAX_CHUNKS;
    if (g > nt) g = nt;
    if (g < 1) g = 1;
    const uint64_t tpc = (nt + g - 1) / g;
    *tiles_per_chunk = uint32_t(tpc < 1 ? 1 : tpc);
    *n_chunks = uint32_t(nt ? (nt + *tiles_per_chunk - 1) / *tiles_per_chunk : 1);
    return cudaSuccess;
}

cudaError_t launch_scan(const Scan8Params& p0, uint64_t alloc_r, cudaStream_t stream) {
    PFN_encodeTiled enc = scan_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    Scan8Params p = p0;
    p.num_tiles = uint32_t(scan_num_tiles(p.n_local));
    const uint32_t kk = p.k > 128u ? 128u : p.k;  // values are <= 127: k >= 128 never matches
    for (int b = 0; b < 7; ++b) p.km[b] = ((kk >> b) & 1u) ? 0xffffffffu : 0u;
    p.km[7] = kk >= 128u ? 0xffffffffu : 0u;
    // tiles [t_int_lo, t_int_hi) need none of the edge rules: not the first tile of the eBWT, wholly inside n_local, not
    // the tile that holds position n_global - 1 nor the one that holds n_global - 2 (an END there decides the post-EOF
    // phantom value; it can be an earlier tile than n_global - 1's, or the last tile of a range that is not the last)
    p.t_int_lo = p.global_off == 0 ? 1u : 0u;
    p.t_int_hi = p.global_off + p.n_local == p.n_global ? (p.num_tiles ? p.num_tiles - 1 : 0) : uint32_t(p.n_local / SC_T);
    if (p.n_global >= 2 && p.n_global - 2 >= p.global_off && p.n_global - 2 < p.global_off + p.n_local) {
        const uint32_t t_nm2 = uint32_t((p.n_global - 2 - p.global_off) / SC_T);
        if (t_nm2 < p.t_int_hi) p.t_int_hi = t_nm2;
    }
    // the bit-sliced LCP as rows of 256 bytes = one run of 32 words (8 rows per block of LCPT_BLOCK positions); the boxes
    // the kernel takes from it are 2 words x 8 runs: the plane words of the group before / after a tile
    CUtensorMap tmap;
    cuuint64_t gdim[2] = {256, cuuint64_t(lcpt_bytes(alloc_r) / 256)};
    cuuint64_t gstride[1] = {256};
    cuuint32_t box[2] = {16, 8};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(p.lcpt), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    int occ = 0;
    const int rc = scan_occupancy(&occ);
    if (rc) return cudaError_t(rc);
    scan_kernel()<<<dim3(p.n_chunks), dim3(SC_THREADS), SC_DYN_SMEM, stream>>>(tmap, p);
    return cudaGetLastError();
}

cudaError_t launch_chunk_resolve(const ResolveParams& p, cudaStream_t stream) {
    if (p.n_chunks > uint32_t(RS_THREADS)) return cudaErrorInvalidValue;
    k_chunk_resolve<<<1, RS_THREADS, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_export_records(const ChunkSeg* segs, uint32_t n_chunks, uint64_t seg_cap, const uint64_t* seg_start,
                                  const uint16_t* seg_len, uint64_t* out_start, uint16_t* out_len, uint8_t* out_packed,
                                  cudaStream_t stream) {
    if (!n_chunks) return cudaSuccess;
    uint64_t bx = (seg_cap + 255) / 256;
    if (bx > 16) bx = 16;
    if (bx < 1) bx = 1;
    k_export_records<<<dim3(unsigned(bx), n_chunks > 1024 ? 1024 : n_chunks), 256, 0, stream>>>(
        segs, n_chunks, seg_cap, seg_start, seg_len, out_start, out_len, reinterpret_cast<uint16_t*>(out_packed));
    return cudaGetLastError();
}

}  // namespace e2s
