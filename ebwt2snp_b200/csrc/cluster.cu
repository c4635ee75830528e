// Phase 1 (ebwt2clust): K1 = streaming LCP boundary stencil, K2 = chunked reduce-then-scan + compaction.
//
// Replaces the sequential state machine of cluster_lm / append_entry (ref:ebwt2clust.cpp:54-139)
// by its local-stencil form (SURVEY.md §8(a) A2):
//   ge(i)    = lcp[i] >= k
//   END(i)   = ge(i) & ( (lcp[i-1] > lcp[i] & lcp[i] <= lcp[i+1]) | !ge(i+1) )        1 <= i <= n-2
//   START(i) = ge(i) & ( !ge(i-1) | END(i-1) )
//   fix-ups  : END(0) = 0;  END(1) = 1 if ge(0) & !ge(1)   (ref:ebwt2clust.cpp:83-84: a cluster opened
//              at 0 is still "open" at 1);  END(n-1) and position n are left to the host tail rule
//              (e2s_cluster_merge), because they depend on the post-EOF phantom record.
//   the j-th START pairs with the j-th END; record = (START, (END-START+1) mod 2^16), kept iff >= min_len.
//
// K1  k_lcp_flags: pure streaming map LCP -> two bit masks (START, END), one bit per position.
//     Persistent CTAs; each 8192-position tile (256 rows x 32 u32) is brought to shared memory by TMA
//     (cp.async.bulk.tensor.2d, hardware 128B swizzle => the blocked per-thread 128-bit reads are bank
//     conflict free), STAGES tiles in flight per CTA behind mbarriers; every thread owns 32 consecutive
//     positions in registers and writes one 32-bit word per mask (a warp writes 128 contiguous bytes).
//     Traffic: 4 B/position read + 0.25 B/position written.  No inter-CTA dependency.
// K2  k_cluster_emit: works on the bit masks only.  One contiguous chunk of 32768-position tiles per CTA:
//     a bit-parallel count pass, ONE exchange of per-chunk values between the CTAs, then the write pass
//     (see the comment above the kernel).  Records come out compacted in position order, 10 B each; their
//     length histogram (statistics(), ref:clust2snp.cpp:899-907) is accumulated on the way.  In fused mode
//     (e2s_cluster_prefilter) the write pass also applies clust2snp's BWT-only prefilter to every record it
//     writes, with range popcounts on the shard's resident base-code bit planes (planes.cuh).

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "internal.h"
#include "planes.cuh"

namespace e2s {

constexpr uint32_t FULL = 0xffffffffu;

// =============================================================================================
// K1: LCP -> START / END bit masks
// =============================================================================================
constexpr int FL_THREADS = 256;
constexpr int FL_V = 32;                      // positions per thread = one 128-byte swizzle row
constexpr int FL_T = FL_THREADS * FL_V;       // 8192 positions per tile

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}

template <int STAGES>
__global__ void __launch_bounds__(FL_THREADS) k_lcp_flags(const __grid_constant__ CUtensorMap tmap, FlagParams p) {
    constexpr int V = FL_V, T = FL_T, CH = V / 4;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t full_bar[STAGES];

    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t k = p.k;
    const uint32_t xr = tid & 7, xr_prev = (tid - 1) & 7, xr_next = (tid + 1) & 7;  // 128B swizzle: chunk ^= row & 7

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&full_bar[s], 1);
        fence_mbar_init();
    }
    __syncthreads();
    const uint32_t num_tiles = p.num_tiles;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            uint64_t t = uint64_t(blockIdx.x) + uint64_t(s) * gridDim.x;
            if (t < num_tiles) {
                mbar_expect_tx(&full_bar[s], T * 4);
                tma_load_2d(tiles + size_t(s) * T * 4, &tmap, 0, int(t * FL_THREADS), &full_bar[s]);
            }
        }
    }

    uint32_t it = 0;
    for (uint64_t t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const int stage = it % STAGES;
        const uint32_t parity = (it / STAGES) & 1;
        const uint64_t tile_base = t * T;
        const uint64_t my_base = tile_base + uint64_t(tid) * V;
        const uint8_t* tile = tiles + size_t(stage) * T * 4;

        uint32_t g_m2 = 0, g_m1 = 0, g_p = 0;  // halo values outside the tile: issue the global loads early
        if (tid == 0) {
            uint2 h = *reinterpret_cast<const uint2*>(p.lcp + (int64_t(tile_base) - 2));
            g_m2 = h.x;
            g_m1 = h.y;
        }
        if (tid == FL_THREADS - 1) g_p = p.lcp[tile_base + T];

        mbar_wait(&full_bar[stage], parity);

        uint32_t v[V];
        {
            const uint8_t* row = tile + size_t(tid) * V * 4;
#pragma unroll
            for (int j = 0; j < CH; ++j) {
                uint4 c = lds128(row + ((uint32_t(j) ^ xr) << 4));
                v[4 * j + 0] = c.x;
                v[4 * j + 1] = c.y;
                v[4 * j + 2] = c.z;
                v[4 * j + 3] = c.w;
            }
        }
        uint32_t v_m2 = __shfl_up_sync(FULL, v[V - 2], 1);
        uint32_t v_m1 = __shfl_up_sync(FULL, v[V - 1], 1);
        uint32_t v_p = __shfl_down_sync(FULL, v[0], 1);
        if (lane == 0) {
            if (tid == 0) {
                v_m2 = g_m2;
                v_m1 = g_m1;
            } else {
                const uint8_t* prow = tile + size_t(tid - 1) * V * 4 + ((uint32_t(CH - 1) ^ xr_prev) << 4);
                uint2 h = *reinterpret_cast<const uint2*>(prow + 8);
                v_m2 = h.x;
                v_m1 = h.y;
            }
        }
        if (lane == 31) {
            if (tid == FL_THREADS - 1) v_p = g_p;
            else v_p = *reinterpret_cast<const uint32_t*>(tile + size_t(tid + 1) * V * 4 + ((0u ^ xr_next) << 4));
        }
        __syncthreads();  // every thread has its tile data in registers: the stage can be refilled
        if (tid == 0) {
            uint64_t tn = t + uint64_t(STAGES) * gridDim.x;
            if (tn < num_tiles) {
                mbar_expect_tx(&full_bar[stage], T * 4);
                tma_load_2d(tiles + size_t(stage) * T * 4, &tmap, 0, int(tn * FL_THREADS), &full_bar[stage]);
            }
        }

        uint32_t G = 0, A = 0;  // G_j = ge(j); A_j = lcp[j-1] > lcp[j]
#pragma unroll
        for (int j = 0; j < V; ++j) {
            G |= uint32_t(v[j] >= k) << j;
            A |= uint32_t((j == 0 ? v_m1 : v[j - 1]) > v[j]) << j;
        }
        const uint32_t g_m1b = v_m1 >= k, g_pb = v_p >= k;
        const uint32_t a_V = v[V - 1] > v_p;
        const uint32_t Gn = (G >> 1) | (g_pb << (V - 1));  // ge(j+1)
        const uint32_t An = (A >> 1) | (a_V << (V - 1));   // lcp[j] > lcp[j+1]
        uint32_t E = G & ((A & ~An) | ~Gn);
        uint32_t e_prev = g_m1b & ((uint32_t(v_m2 > v_m1) & ((~A) & 1u)) | ((~G) & 1u));

        const uint64_t gpos = p.global_off + my_base;
        if (gpos == 0) {  // the init special cases of ref:ebwt2clust.cpp:83-86
            E &= ~1u;
            e_prev = 0;
            if ((G & 1u) && !(G & 2u)) E |= 2u;
        }
        uint32_t vm;
        {
            const int64_t nvalid = int64_t(p.n_local) - int64_t(my_base);
            vm = nvalid >= V ? FULL : (nvalid <= 0 ? 0u : ((1u << nvalid) - 1u));
            const int64_t last = int64_t(p.n_global) - 1 - int64_t(gpos);  // END(n_global-1): host tail rule
            if (last >= 0 && last < V) E &= ~(1u << last);
        }
        E &= vm;
        const uint32_t Gp = (G << 1) | g_m1b;
        const uint32_t Ep = (E << 1) | e_prev;
        const uint32_t S = G & (~Gp | Ep) & vm;

        const uint64_t w = t * FL_THREADS + tid;
        p.s_words[w] = S;
        p.e_words[w] = E;
    }
}

// =============================================================================================
// K2: chunked reduce-then-scan over the bit masks + compaction
// =============================================================================================
// START and END bits alternate (S <= E < S' <= E' ...): every END closes the cluster opened by the nearest
// START at or before it.  The grid cuts the shard's mask words into one contiguous CHUNK per CTA and makes
// two passes over its chunk with ONE exchange in between, so no tile ever waits for another tile:
//   pass 1  counts the records the chunk will keep.  Which ENDs are dropped by the min_len test is a
//           bit-parallel function of the masks (a START within min_len - 1 positions, min_len <= 33), so
//           this is a pure streaming popcount pass (no barriers except one vote per tile, see `flagged`).
//   exchange every CTA publishes (kept count, first/last START and END of the chunk) -- values that do not
//           depend on any other chunk -- resolves the one END that may close a cluster opened in an earlier
//           chunk (exact wrapped-length test), publishes its final count and sums the final counts of the
//           chunks before it: depth-2 dependency, no chain.
//   pass 2  re-reads the chunk (L2), scatters the END positions with their output ranks into shared memory
//           and writes the records with one lane per record: the START is found by a backward search in the
//           tile's START mask (shared memory), offsets are running sums inside the CTA.
// Exactness: the bit-parallel count is exact unless the wrapped length (L mod 2^16) matters, i.e. a cluster
// is >= 65503 long.  Such a cluster implies >= 7 of the 8 warps of some tile see no event at all; pass 1
// votes on that per tile and the chunk then falls back to the EXACT routine (also used for min_len > 33),
// which pairs and tests every END individually in both passes.
constexpr int EM_THREADS = 256;
constexpr int EM_WARPS = EM_THREADS / 32;
constexpr int EM_WPT = 4;                               // 32-bit words per thread and mask (one uint4)
constexpr int EM_TILE_WORDS = EM_THREADS * EM_WPT;      // 1024 words = 32768 positions
constexpr int EM_TILE_POS = EM_TILE_WORDS * 32;
constexpr int EM_CAP = 2048;                            // ENDs per scatter window
constexpr int EM_PF_QUADS = EM_TILE_POS / 64 + PL_PAD / 64;  // plane quads of one tile and of the PL_PAD positions before it
constexpr int EM_DESC_WORDS = 8;                        // u64 words per chunk descriptor
constexpr int EM_MAX_CHUNKS = 148 * 8 * 2;              // upper bound of the grid (descriptor allocation)

// payload encoding of the open-cluster state
constexpr uint64_t OPEN_NONE = 0;
constexpr uint64_t OPEN_UNKNOWN = 1;  // open or not is decided by an earlier shard
constexpr uint64_t OPEN_BIAS = 2;     // payload = global start + 2

// chunk descriptor words
enum { CD_A = 0, CD_FIRST_E = 1, CD_FIRST_S = 2, CD_LAST_S = 3, CD_LAST_E = 4, CD_B = 5 };
constexpr uint64_t CD_VALID = uint64_t(1) << 63;

__device__ __forceinline__ void st_release(uint64_t* p, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t wait_valid(const uint64_t* p) {
    uint64_t v;
    while (!((v = ld_acquire(p)) & CD_VALID)) __nanosleep(40);
    return v;
}

// the wrapped length test of append_entry (ref:ebwt2clust.cpp:56,104)
__device__ __forceinline__ bool keep_len(uint64_t st, uint64_t gend, int32_t min_len, uint32_t* len) {
    *len = uint32_t(gend - st + 1) & 0xffffu;
    return int(*len) >= min_len;
}

// highest / lowest set bit of a 128-bit value held in 4 words (word 0 = lowest positions); -1 / 128 if none
__device__ __forceinline__ int top_bit128(const uint32_t w[4]) {
    const unsigned long long hi = (uint64_t(w[3]) << 32) | w[2], lo = (uint64_t(w[1]) << 32) | w[0];
    return hi ? 127 - __clzll(hi) : (lo ? 63 - __clzll(lo) : -1);
}
__device__ __forceinline__ int low_bit128(const uint32_t w[4]) {
    const unsigned long long hi = (uint64_t(w[3]) << 32) | w[2], lo = (uint64_t(w[1]) << 32) | w[0];
    return lo ? __ffsll(lo) - 1 : (hi ? 63 + __ffsll(hi) : 128);
}

struct EmitShared {
    uint32_t smask[EM_TILE_WORDS];  // START mask of the tile (backward search for the START of an END)
    uint32_t emask[EM_TILE_WORDS];  // END mask of the tile
    uint16_t ek[EM_CAP];            // ek[q] = tile-local position of the tile's (win + q)-th listed END (bit-parallel mode: kept ENDs only)
    uint32_t wsum[EM_WARPS];        // per warp: #END | #dropped << 16
    alignas(8) uint8_t wev[2][EM_WARPS];  // pass 1: per warp, bit 0 = has a START, bit 1 = has an END (double buffered)
    uint8_t wfirst_end[EM_WARPS];         // pass 1, rare path: the warp's first event is an END
    int t_last_s, t_last_e, t_first_s, t_first_e;  // tile-local positions, -1 / NO_POS = none (written by warp 0)
    uint32_t row_kept;              // EXACT: running kept count of the tile
    unsigned long long red[6];      // block reductions of pass 1
    uint64_t x_in, prefix, carried_pos;
    uint32_t adj;
    unsigned int hist[E2S_HIST_BINS];
};

constexpr int NO_POS = 0x7fffffff;
constexpr uint64_t NO_TILE = ~0ull;

__device__ __forceinline__ bool has_zero_byte(uint32_t x) { return ((x - 0x01010101u) & ~x & 0x80808080u) != 0; }

__global__ void __launch_bounds__(EM_THREADS, 4) k_cluster_emit(EmitParams p) {
    __shared__ EmitShared sh;
    __shared__ unsigned long long s_chunk;
    __shared__ __align__(16) uint4 pf_win[EM_PF_QUADS];  // fused prefilter: the tile's window of the resident bit planes
    __shared__ uint64_t pf_bar;
    const bool pf = p.pf_mcov != 0;
    uint32_t pf_parity = 0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int spread = p.min_len >= 2 ? p.min_len - 2 : -1;  // extra positions a START shadows; -1: nothing is dropped

    for (int i = tid; i < E2S_HIST_BINS; i += EM_THREADS) sh.hist[i] = 0;
    if (pf && tid == 0) {
        mbar_init(&pf_bar, 1);
        fence_mbar_init();
    }
    // Chunks are handed out by a ticket, so every chunk with a smaller id is owned by a CTA that is already
    // running: the spin-waits of the exchange cannot deadlock whatever else occupies the SMs.
    if (tid == 0) s_chunk = atomicAdd(&p.res->ticket, 1ull);
    __syncthreads();
    const uint64_t c = s_chunk, n_chunks = gridDim.x;
    const uint64_t tpc = (p.num_tiles + n_chunks - 1) / n_chunks;  // tiles per chunk
    const uint64_t t_lo = c * tpc < p.num_tiles ? c * tpc : p.num_tiles;
    const uint64_t t_hi = t_lo + tpc < p.num_tiles ? t_lo + tpc : p.num_tiles;
    uint64_t* my_desc = p.desc + c * EM_DESC_WORDS;
    bool exact = p.min_len > 33;  // CTA-uniform

    // D = ENDs of clusters shorter than min_len: a START at the same position or up to `spread` positions before.
    // `pv` = START word preceding S[0] (0 at the start of the chunk: an END shadowed from an earlier chunk is the
    // chunk's first END, which the exchange tests exactly).
    auto dropped_mask = [&](const uint32_t S[EM_WPT], const uint32_t E[EM_WPT], uint32_t pv, uint32_t D[EM_WPT]) {
#pragma unroll
        for (int j = 0; j < EM_WPT; ++j) {
            uint32_t sp = 0;
            if (spread >= 0) {
                sp = S[j];
                const uint32_t prev = j ? S[j - 1] : pv;
                for (int d = 1; d <= spread; ++d) sp |= __funnelshift_l(prev, S[j], d);
            }
            D[j] = E[j] & sp;
        }
    };
    auto prev_word = [&](uint64_t t, uint64_t word0, uint32_t my_last_word) -> uint32_t {
        if (spread <= 0) return 0u;  // uniform: only the shifted copies look at the previous word
        uint32_t pv = __shfl_up_sync(FULL, my_last_word, 1);
        if (lane == 0) pv = (tid == 0 && t == t_lo) ? 0u : __ldg(p.s_words + word0 - 1);
        return pv;
    };
    // global position of the first / last set bit of `mask` inside tile t (block-wide; ~0 / 0 = none; last is 1 + position)
    auto locate = [&](const uint32_t* mask, uint64_t t, bool want_first) -> unsigned long long {
        __syncthreads();
        if (tid == 0) sh.red[0] = want_first ? ~0ull : 0ull;
        __syncthreads();
        if (t != NO_TILE) {
            const uint4 m4 = __ldg(reinterpret_cast<const uint4*>(mask + t * EM_TILE_WORDS + uint64_t(tid) * EM_WPT));
            const uint32_t M[EM_WPT] = {m4.x, m4.y, m4.z, m4.w};
            const uint64_t gbase = p.global_off + t * uint64_t(EM_TILE_POS) + uint64_t(tid) * (EM_WPT * 32);
            if (want_first) {
                const int b = low_bit128(M);
                if (b < 128) atomicMin(&sh.red[0], (unsigned long long)(gbase + b));
            } else {
                const int b = top_bit128(M);
                if (b >= 0) atomicMax(&sh.red[0], (unsigned long long)(gbase + b + 1));
            }
        }
        __syncthreads();
        return sh.red[0];
    };

    // ================= pass 1 (bit-parallel): kept count, first / last events of the chunk =================
    unsigned long long kept_prov = 0, n_end_chunk = 0;
    unsigned long long first_e = ~0ull, first_s = ~0ull, last_s = 0, last_e = 0;  // first: global position; last: 1 + global position
    if (!exact) {
        uint32_t kept_t = 0, ends_t = 0;
        uint64_t ft_s = NO_TILE, ft_e = NO_TILE, lt_s = NO_TILE, lt_e = NO_TILE;  // first / last tile in which my warp saw a START / END
        bool flagged = false, seen = false;
        uint32_t run = 0;  // consecutive 4096-position blocks without any event (block-uniform)
        uint4 s4 = make_uint4(0, 0, 0, 0), e4 = s4;
        if (t_lo < t_hi) {
            const uint64_t w0 = t_lo * EM_TILE_WORDS + uint64_t(tid) * EM_WPT;
            s4 = __ldg(reinterpret_cast<const uint4*>(p.s_words + w0));
            e4 = __ldg(reinterpret_cast<const uint4*>(p.e_words + w0));
        }
        for (uint64_t t = t_lo; t < t_hi; ++t) {
            const uint64_t word0 = t * EM_TILE_WORDS + uint64_t(tid) * EM_WPT;
            const uint32_t S[EM_WPT] = {s4.x, s4.y, s4.z, s4.w};
            const uint32_t E[EM_WPT] = {e4.x, e4.y, e4.z, e4.w};
            if (t + 1 < t_hi) {  // next tile's loads stay in flight across the barrier
                s4 = __ldg(reinterpret_cast<const uint4*>(p.s_words + word0 + EM_TILE_WORDS));
                e4 = __ldg(reinterpret_cast<const uint4*>(p.e_words + word0 + EM_TILE_WORDS));
            }
            uint32_t D[EM_WPT];
            dropped_mask(S, E, prev_word(t, word0, S[EM_WPT - 1]), D);
            uint32_t ce = 0, cd = 0;
#pragma unroll
            for (int j = 0; j < EM_WPT; ++j) {
                ce += __popc(E[j]);
                cd += __popc(D[j]);
            }
            ends_t += ce;
            kept_t += ce - cd;
            const bool any_s = __any_sync(FULL, (S[0] | S[1] | S[2] | S[3]) != 0), any_e = __any_sync(FULL, ce != 0);
            if (any_s) {
                lt_s = t;
                if (ft_s == NO_TILE) ft_s = t;
            }
            if (any_e) {
                lt_e = t;
                if (ft_e == NO_TILE) ft_e = t;
            }
            // Wrap watch: a cluster of >= 65503 positions leaves >= 14 consecutive aligned 4096-position blocks (one
            // per warp and tile) without any event between its START and its END.
            if (lane == 0) sh.wev[t & 1][warp] = uint8_t(uint32_t(any_s) | (uint32_t(any_e) << 1));
            __syncthreads();
            const uint2 ev = *reinterpret_cast<const uint2*>(sh.wev[t & 1]);
            if (run == 0 && !has_zero_byte(ev.x) && !has_zero_byte(ev.y)) {  // every warp saw an event: the usual case
                run = 0;
                seen = true;
            } else {
                // rare (block-uniform): some 4096-position block is empty or a run of empty blocks is pending.  A run matters
                // only if it lies INSIDE a cluster, i.e. the first event after it is an END that no START precedes.
                {
                    const int fs = low_bit128(S), fe = low_bit128(E);
                    const int wfs = __reduce_min_sync(FULL, fs < 128 ? lane * 128 + fs : NO_POS);
                    const int wfe = __reduce_min_sync(FULL, fe < 128 ? lane * 128 + fe : NO_POS);
                    if (lane == 0) sh.wfirst_end[warp] = uint8_t(wfe < wfs);
                }
                __syncthreads();
                for (int w = 0; w < EM_WARPS; ++w) {
                    const uint32_t b = ((w < 4 ? ev.x : ev.y) >> (8 * (w & 3))) & 0xffu;
                    if (!b) {
                        ++run;
                    } else {
                        if (run >= 14 && seen && sh.wfirst_end[w]) flagged = true;
                        run = 0;
                        seen = true;
                    }
                }
            }
        }
        if (flagged) {
            exact = true;  // a cluster may be long enough for its 16-bit length to wrap: count exactly below
        } else {
            if (tid < 6) sh.red[tid] = (tid == 2 || tid == 3) ? ~0ull : 0ull;
            __syncthreads();
            const uint32_t wk = __reduce_add_sync(FULL, kept_t), we = __reduce_add_sync(FULL, ends_t);
            if (lane == 0) {
                atomicAdd(&sh.red[0], (unsigned long long)wk);
                atomicAdd(&sh.red[1], (unsigned long long)we);
                if (ft_e != NO_TILE) atomicMin(&sh.red[2], (unsigned long long)ft_e);
                if (ft_s != NO_TILE) atomicMin(&sh.red[3], (unsigned long long)ft_s);
                if (lt_s != NO_TILE) atomicMax(&sh.red[4], (unsigned long long)lt_s + 1);
                if (lt_e != NO_TILE) atomicMax(&sh.red[5], (unsigned long long)lt_e + 1);
            }
            __syncthreads();
            kept_prov = sh.red[0];
            n_end_chunk = sh.red[1];
            const uint64_t tfe = sh.red[2], tfs = sh.red[3], tls = sh.red[4], tle = sh.red[5];
            // exact positions of the chunk's first / last START and END: one look at the four tiles that hold them
            first_e = locate(p.e_words, tfe, true);
            first_s = locate(p.s_words, tfs, true);
            last_s = locate(p.s_words, tls ? tls - 1 : NO_TILE, false);
            last_e = locate(p.e_words, tle ? tle - 1 : NO_TILE, false);
        }
    }

    // ================= the tile routine: pass 2, and pass 1 of EXACT chunks =================
    // Processes tile t with the open state X entering it; updates X to the state leaving the tile and returns the
    // tile's kept count (block-uniform).  write: records go to out[obase + rank].
    //   carried_pos : global position of the chunk's first END if its START lies before the chunk (known after
    //                 the exchange), ~0 otherwise;  adj = 1 if that END turned out not to be kept
    //   resolved    : X is authoritative (false in pass 1 of an EXACT chunk until an event has been seen)
    unsigned long long acc_bases = 0;
    struct TileInfo { int first_s, first_e, last_s, last_e; uint32_t n_end; };
    auto tile_pass = [&](uint64_t t, uint64_t& X, bool resolved, uint64_t obase, bool write, uint64_t carried_pos,
                         uint32_t adj, uint64_t chunk_end, TileInfo* info) -> uint32_t {
        __syncthreads();  // shared state of the previous tile is no longer read
        const uint64_t word0 = t * EM_TILE_WORDS + uint64_t(tid) * EM_WPT;
        const uint4 s4 = __ldg(reinterpret_cast<const uint4*>(p.s_words + word0));
        const uint4 e4 = __ldg(reinterpret_cast<const uint4*>(p.e_words + word0));
        const uint32_t S[EM_WPT] = {s4.x, s4.y, s4.z, s4.w};
        const uint32_t E[EM_WPT] = {e4.x, e4.y, e4.z, e4.w};
        const uint64_t tile_gbase = p.global_off + t * uint64_t(EM_TILE_POS);
        const bool pf_tile = pf && write;
        bool pf_pending = pf_tile;  // the window has been requested and not yet waited for (block-uniform)
        if (pf_tile && tid == 0) {  // plane quads of the tile and of the 192 positions before it, by the bulk-copy engine
            fence_proxy_async();    // the previous tile's window was read through the generic proxy
            mbar_expect_tx(&pf_bar, EM_PF_QUADS * 16);
            bulk_g2s(pf_win, p.planes + t * uint64_t(EM_TILE_POS / 64), EM_PF_QUADS * 16, &pf_bar);
        }
        auto pf_wait = [&]() {
            if (pf_pending) {
                mbar_wait(&pf_bar, pf_parity);
                pf_parity ^= 1u;
                pf_pending = false;
            }
        };
        reinterpret_cast<uint4*>(sh.smask)[tid] = s4;
        reinterpret_cast<uint4*>(sh.emask)[tid] = e4;
        uint32_t D[EM_WPT] = {0, 0, 0, 0};
        if (!exact) dropped_mask(S, E, prev_word(t, word0, S[EM_WPT - 1]), D);
        uint32_t cE = 0, cD = 0;
#pragma unroll
        for (int j = 0; j < EM_WPT; ++j) {
            cE += __popc(E[j]);
            cD += __popc(D[j]);
        }
        const uint32_t pk = cE | (cD << 16);
        uint32_t inc = pk;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(FULL, inc, d);
            if (lane >= d) inc += o;
        }
        if (lane == 31) sh.wsum[warp] = inc;
        if (tid == 0) sh.row_kept = 0;
        __syncthreads();  // (1) masks and the per-warp sums
        if (warp == 0) {
            // last (and, for pass 1 of an EXACT chunk, first) START / END of the tile: warp-wide search in the shared masks
            auto top_of = [&](const uint32_t* m) -> int {
                for (int b0 = EM_TILE_WORDS - 32; b0 >= 0; b0 -= 32) {
                    const uint32_t w = m[b0 + lane];
                    const uint32_t bal = __ballot_sync(FULL, w != 0);
                    if (bal) {
                        const int hl = 31 - __clz(bal);
                        return (b0 + hl) * 32 + 31 - __clz(__shfl_sync(FULL, w, hl));
                    }
                }
                return -1;
            };
            auto low_of = [&](const uint32_t* m) -> int {
                for (int b0 = 0; b0 < EM_TILE_WORDS; b0 += 32) {
                    const uint32_t w = m[b0 + lane];
                    const uint32_t bal = __ballot_sync(FULL, w != 0);
                    if (bal) {
                        const int ll = __ffs(bal) - 1;
                        return (b0 + ll) * 32 + __ffs(__shfl_sync(FULL, w, ll)) - 1;
                    }
                }
                return NO_POS;
            };
            const int ls = top_of(sh.smask), le = top_of(sh.emask);
            int fs = NO_POS, fe = NO_POS;
            if (info) {
                fs = low_of(sh.smask);
                fe = low_of(sh.emask);
            }
            if (lane == 0) {
                sh.t_last_s = ls;
                sh.t_last_e = le;
                sh.t_first_s = fs;
                sh.t_first_e = fe;
            }
        }
        uint32_t base = inc - pk, tot = 0;
#pragma unroll
        for (int q = 0; q < EM_WARPS; ++q) {
            const uint32_t ws = sh.wsum[q];
            if (q < warp) base += ws;
            tot += ws;
        }
        const uint32_t nE = tot & 0xffffu, nD = tot >> 16;
        const uint32_t myEbase = base & 0xffffu, myDbase = base >> 16;
        const bool carried_here = carried_pos - tile_gbase < uint64_t(EM_TILE_POS);  // the chunk's carried-in END lies in this tile

        // START of the cluster closed by the END at tile-local position e: nearest START bit at or before e
        auto find_start = [&](uint32_t e, bool* in_tile, bool* known) -> uint64_t {
            int w = int(e >> 5);
            uint32_t m = sh.smask[w] & ((2u << (e & 31)) - 1u);
            while (!m && w > 0) m = sh.smask[--w];
            *in_tile = m != 0;
            *known = true;
            if (m) return tile_gbase + uint32_t(w) * 32u + uint32_t(31 - __clz(m));
            *known = X >= OPEN_BIAS;
            return X - OPEN_BIAS;
        };

        // fused prefilter of find_variants on a record just written at index o (ref:clust2snp.cpp:402-429, planes.cuh)
        auto prefilter = [&](uint64_t st, uint32_t len, uint64_t o) {
            if (len < 2 * p.pf_mcov || len > uint32_t(MAX_C_LEN)) return;
            // clust2snp analyses the positions [st, st + len) with the WRAPPED 16-bit length: for a cluster of 65536 + len
            // positions that range lies far before this tile's window -- leave the decision to the exact test
            if (st + PL_PAD < tile_gbase ||
                frequent_codes<false>(pf_win, int64_t(st) - int64_t(tile_gbase), len, p.pf_mcov) >= 2) {
                const unsigned long long at = atomicAdd(&p.res->n_pf, 1ull);
                if (at < p.pf_cap) p.pf_list[at] = SurvEntry{st, st - p.global_off, len, 0u};
                        else p.res->overflow |= 2;  // (seen by every rank in the exchange rows: all of them repeat the round)
            }
        };
        // The list holds the ENDs that will be written: all of them in EXACT mode (D = 0), the kept ones otherwise
        // (the carried-in END counts as kept until the exchange has tested it).
        const uint32_t nL = nE - nD, cL = cE - cD, myLbase = myEbase - myDbase;
        if (write && !exact && nD && p.n_global - 2 - tile_gbase < uint64_t(EM_TILE_POS)) {
            // A dropped END at position n_global - 2 still decides the reference's post-EOF phantom value (SURVEY.md A3).
            const uint32_t e = uint32_t(p.n_global - 2 - tile_gbase);
            if (tid == 0 && ((sh.emask[e >> 5] >> (e & 31)) & 1u)) {
                bool in_tile, known;
                const uint64_t st = find_start(e, &in_tile, &known);
                p.res->end_nm2_start = known ? st + 1 : ~0ull;
            }
        }
        for (uint32_t win = 0; win < nL; win += EM_CAP) {  // one iteration unless the tile lists > EM_CAP ENDs
            if (win) __syncthreads();  // the previous window's list is no longer read
            if (myLbase < win + EM_CAP && myLbase + cL > win) {
                uint32_t ord = myLbase - win;  // may wrap below 0: the unsigned compare rejects those
#pragma unroll
                for (int h = 0; h < EM_WPT / 2; ++h) {
                    unsigned long long m = (uint64_t(E[2 * h + 1] & ~D[2 * h + 1]) << 32) | (E[2 * h] & ~D[2 * h]);
                    while (m) {
                        const int b = __ffsll(m) - 1;
                        m &= m - 1;
                        if (ord < EM_CAP) sh.ek[ord] = uint16_t((tid * EM_WPT + 2 * h) * 32 + b);
                        ++ord;
                    }
                }
            }
            __syncthreads();  // (2) list
            pf_wait();
            const uint32_t cntw = nL - win < EM_CAP ? nL - win : EM_CAP;
            if (!exact) {
                if (!write) continue;
                // dense pass: one lane per kept END; its rank in the tile is its place in the list
                for (uint32_t q = tid; q < cntw; q += EM_THREADS) {
                    const uint32_t e = sh.ek[q];
                    const uint64_t gend = tile_gbase + e;
                    uint32_t r = win + q;
                    bool in_tile, known;
                    const uint64_t st = find_start(e, &in_tile, &known);
                    uint32_t len = uint32_t(gend - st + 1) & 0xffffu;  // (no wrap unless carried in: a bit-parallel chunk has no cluster >= 65503)
                    if (gend == carried_pos) {  // resolved by the exchange (exact wrapped-length test)
                        if (gend + 2 == p.n_global) p.res->end_nm2_start = known ? st + 1 : ~0ull;
                        if (!known) {           // the shard's head END: its START is in an earlier shard
                            p.res->head_end = gend + 1;
                            continue;
                        }
                        if (adj) continue;      // not kept after all
                    } else {
                        if (carried_here) r -= adj;
                        if (gend + 2 == p.n_global) p.res->end_nm2_start = st + 1;
                    }
                    const uint64_t o = obase + r;
                    if (o < p.cap) {
                        p.out_start[o] = st;
                        p.out_len[o] = uint16_t(len);
                    } else {
                        p.res->overflow |= 1;
                    }
                    acc_bases += len;
                    if (len <= MAX_C_LEN) atomicAdd(&sh.hist[len], 1u);
                    if (o + 1 == chunk_end) atomicMax(&p.res->last_rec, (unsigned long long)(((o + 1) << 16) | len));
                    if (pf_tile) prefilter(st, len, o);
                }
            } else if (warp == 0) {
                // EXACT: one warp pairs, tests and ranks every END in order (min_len > 33, or a very long cluster nearby)
                uint32_t running = sh.row_kept;
                for (uint32_t q0 = 0; q0 < cntw; q0 += 32) {
                    const uint32_t q = q0 + lane;
                    bool k = false, head = false;
                    uint64_t st = 0, gend = 0;
                    uint32_t len = 0;
                    if (q < cntw) {
                        const uint32_t e = sh.ek[q];
                        gend = tile_gbase + e;
                        bool in_tile, known;
                        st = find_start(e, &in_tile, &known);
                        if (!in_tile && !resolved) k = true;  // the chunk's first END before the exchange: provisional, fixed there
                        else if (!known) head = true;
                        else k = keep_len(st, gend, p.min_len, &len);
                    }
                    const uint32_t bal = __ballot_sync(FULL, k);
                    if (write && q < cntw) {
                        if (head) {
                            p.res->head_end = gend + 1;
                            if (gend + 2 == p.n_global) p.res->end_nm2_start = ~0ull;
                        } else {
                            if (gend + 2 == p.n_global) p.res->end_nm2_start = st + 1;
                            if (k) {
                                const uint64_t o = obase + running + __popc(bal & ((1u << lane) - 1u));
                                if (o < p.cap) {
                                    p.out_start[o] = st;
                                    p.out_len[o] = uint16_t(len);
                                } else {
                                    p.res->overflow |= 1;
                                }
                                acc_bases += len;
                                if (len <= MAX_C_LEN) atomicAdd(&sh.hist[len], 1u);
                                if (o + 1 == chunk_end) atomicMax(&p.res->last_rec, (unsigned long long)(((o + 1) << 16) | len));
                                if (pf_tile) prefilter(st, len, o);
                            }
                        }
                    }
                    running += __popc(bal);
                }
                if (lane == 0) sh.row_kept = running;
            }
        }
        if (exact || nL == 0) __syncthreads();  // row_kept / warp 0's tile summary (otherwise ordered by barrier (2))
        pf_wait();  // a tile without ENDs: keep the barrier's phase in step with the requests
        const uint32_t tile_kept = exact ? sh.row_kept : nL - (carried_here ? adj : 0u);
        const int t_last_s = sh.t_last_s, t_last_e = sh.t_last_e;
        if (info) {
            info->last_s = t_last_s;
            info->last_e = t_last_e;
            info->first_s = sh.t_first_s;
            info->first_e = sh.t_first_e;
            info->n_end = nE;
        }
        if (t_last_s >= 0 || t_last_e >= 0)  // state leaving the tile
            X = t_last_s > t_last_e ? tile_gbase + uint64_t(t_last_s) + OPEN_BIAS : OPEN_NONE;
        return tile_kept;
    };

    // ================= pass 1 of EXACT chunks =================
    if (exact) {
        uint64_t X = OPEN_UNKNOWN;  // unresolved until the exchange: an END without START so far is the chunk's first END
        bool seen = false;
        kept_prov = 0;
        n_end_chunk = 0;
        first_e = first_s = ~0ull;
        last_s = last_e = 0;
        for (uint64_t t = t_lo; t < t_hi; ++t) {
            TileInfo ti;
            kept_prov += tile_pass(t, X, seen, 0, false, ~0ull, 0, ~0ull, &ti);
            const uint64_t tile_gbase = p.global_off + t * uint64_t(EM_TILE_POS);
            n_end_chunk += ti.n_end;
            if (ti.last_s >= 0) last_s = tile_gbase + uint64_t(ti.last_s) + 1;
            if (ti.last_e >= 0) last_e = tile_gbase + uint64_t(ti.last_e) + 1;
            if (first_e == ~0ull && ti.first_e != NO_POS) first_e = tile_gbase + uint64_t(ti.first_e);
            if (first_s == ~0ull && ti.first_s != NO_POS) first_s = tile_gbase + uint64_t(ti.first_s);
            if (ti.last_s >= 0 || ti.last_e >= 0) seen = true;
        }
    }

    // ================= exchange =================
    if (warp == 0) {
        if (lane == 0) {
            my_desc[CD_FIRST_E] = first_e;
            my_desc[CD_FIRST_S] = first_s;
            my_desc[CD_LAST_S] = last_s;
            my_desc[CD_LAST_E] = last_e;
            st_release(&my_desc[CD_A], CD_VALID | kept_prov);
        }
        // open state entering the chunk: the nearest earlier chunk that has any event decides
        uint64_t X = p.global_off == 0 ? OPEN_NONE : OPEN_UNKNOWN;
        for (int64_t j = int64_t(c) - 1; j >= 0; --j) {
            const uint64_t* d = p.desc + uint64_t(j) * EM_DESC_WORDS;
            wait_valid(d + CD_A);
            const uint64_t ls = desc_load(d + CD_LAST_S), le = desc_load(d + CD_LAST_E);
            if (ls | le) {
                X = ls > le ? (ls - 1) + OPEN_BIAS : OPEN_NONE;
                break;
            }
        }
        // the chunk's first END closes a cluster opened before the chunk iff no START precedes it in the chunk
        const bool carried = first_e != ~0ull && (first_s == ~0ull || first_e < first_s);
        if (X == OPEN_UNKNOWN && !carried && (first_e != ~0ull || first_s != ~0ull)) X = OPEN_NONE;  // the chunk starts with a START
        uint32_t adj = 0;
        if (carried) {
            uint32_t len;
            const bool k = X >= OPEN_BIAS && keep_len(X - OPEN_BIAS, first_e, p.min_len, &len);
            adj = k ? 0u : 1u;
        }
        const uint64_t kept_final = kept_prov - adj;
        if (lane == 0) st_release(&my_desc[CD_B], CD_VALID | kept_final);
        // records kept by the chunks before mine
        uint64_t acc = 0;
        for (int64_t j0 = int64_t(c) - 1 - lane; j0 >= 0; j0 -= 32 * 4) {  // 4 loads in flight per lane; the count sits in the polled word
            uint64_t v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t j = j0 - 32 * u;
                v[u] = j >= 0 ? desc_load(p.desc + uint64_t(j) * EM_DESC_WORDS + CD_B) : CD_VALID;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t j = j0 - 32 * u;
                while (!(v[u] & CD_VALID)) {
                    __nanosleep(40);
                    v[u] = desc_load(p.desc + uint64_t(j) * EM_DESC_WORDS + CD_B);
                }
                acc += v[u] & ~CD_VALID;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
        if (lane == 0) {
            sh.x_in = X;
            sh.prefix = acc;
            sh.adj = adj;
            sh.carried_pos = carried ? first_e : ~0ull;
            sh.red[0] = kept_final;
            atomicAdd(&p.res->n_written, (unsigned long long)kept_final);
            if (n_end_chunk) atomicAdd(&p.res->n_end, n_end_chunk);
            if (last_s | last_e) atomicOr(&p.res->any_event, 1ull);
        }
    }
    __syncthreads();

    // ================= pass 2 =================
    {
        uint64_t X = sh.x_in, obase = sh.prefix;
        const uint64_t chunk_end = sh.prefix + sh.red[0], carried_pos = sh.carried_pos;
        const uint32_t adj = sh.adj;
        for (uint64_t t = t_lo; t < t_hi; ++t) obase += tile_pass(t, X, true, obase, true, carried_pos, adj, chunk_end, nullptr);
        if (c == n_chunks - 1 && tid == 0)  // state after the whole shard
            p.res->open_start = X >= OPEN_BIAS ? X - OPEN_BIAS + 1 : 0;
    }

#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc_bases += __shfl_xor_sync(FULL, acc_bases, d);
    if (lane == 0 && acc_bases) atomicAdd(&p.res->n_bases, acc_bases);
    __syncthreads();
    for (int i = tid; i < E2S_HIST_BINS; i += EM_THREADS)
        if (sh.hist[i]) atomicAdd(&p.res->hist[i], (unsigned long long)sh.hist[i]);
    if (c == 0 && tid == 0 && p.tail_lcp) {
        p.res->tail_lcp_nm2 = p.tail_lcp[0];
        p.res->tail_lcp_nm1 = p.tail_lcp[1];
        p.res->tail_bwt_nm1 = p.tail_bwt[0];
    }
}

// ---- tiny list helpers -----------------------------------------------------------------------
struct PutArgs {
    uint64_t st[3];
    uint64_t ln[3];
    int n;
};
__global__ void k_put_records(uint64_t* d_start, uint16_t* d_len, uint64_t at, PutArgs a) {
    if (int(threadIdx.x) < a.n) {
        d_start[at + threadIdx.x] = a.st[threadIdx.x];
        d_len[at + threadIdx.x] = uint16_t(a.ln[threadIdx.x]);
    }
}
cudaError_t launch_put_records(uint64_t* d_start, uint16_t* d_len, uint64_t at, const uint64_t* st, const uint64_t* ln,
                               int n, cudaStream_t stream) {
    PutArgs a;
    a.n = n;
    for (int i = 0; i < 3; ++i) {
        a.st[i] = i < n ? st[i] : 0;
        a.ln[i] = i < n ? ln[i] : 0;
    }
    k_put_records<<<1, 32, 0, stream>>>(d_start, d_len, at, a);
    return cudaGetLastError();
}

// .clusters file layout: u64 start LE + u16 length LE = 10 bytes, no padding (ref:ebwt2clust.cpp:58-59)
__global__ void k_pack_records(const uint64_t* __restrict__ st, const uint16_t* __restrict__ ln, uint64_t m,
                               uint16_t* __restrict__ out) {
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < m; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint64_t s = st[i];
        uint16_t* o = out + i * 5;
        o[0] = uint16_t(s);
        o[1] = uint16_t(s >> 16);
        o[2] = uint16_t(s >> 32);
        o[3] = uint16_t(s >> 48);
        o[4] = ln[i];
    }
}
cudaError_t launch_pack_records(const uint64_t* d_start, const uint16_t* d_len, uint64_t m, uint8_t* d_out,
                                cudaStream_t stream, int sm_count) {
    if (m == 0) return cudaSuccess;
    uint64_t blocks = (m + 255) / 256;
    if (blocks > uint64_t(sm_count) * 16) blocks = uint64_t(sm_count) * 16;
    k_pack_records<<<unsigned(blocks), 256, 0, stream>>>(d_start, d_len, m, reinterpret_cast<uint16_t*>(d_out));
    return cudaGetLastError();
}

// =============================================================================================
// host side
// =============================================================================================
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
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

uint64_t flags_words_needed(uint64_t n_local) {
    // K1 writes whole 8192-position tiles; K2 reads whole 65536-position tiles
    const uint64_t w = (n_local + 31) / 32;
    return (w + EM_TILE_WORDS - 1) / EM_TILE_WORDS * EM_TILE_WORDS;
}

uint64_t emit_num_tiles(uint64_t n_local) { return flags_words_needed(n_local) / EM_TILE_WORDS; }

cudaError_t launch_flags(const FlagParams& p0, uint64_t rows_alloc32, int sm_count, cudaStream_t stream) {
    constexpr int STAGES = 3;  // LCP tiles in flight per CTA
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    FlagParams p = p0;
    p.num_tiles = uint32_t((p.n_local + FL_T - 1) / FL_T);
    CUtensorMap tmap;
    cuuint64_t gdim[2] = {cuuint64_t(FL_V), cuuint64_t(rows_alloc32)};
    cuuint64_t gstride[1] = {cuuint64_t(FL_V) * 4};
    cuuint32_t box[2] = {cuuint32_t(FL_V), cuuint32_t(FL_THREADS)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<uint32_t*>(p.lcp), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    const size_t smem = size_t(STAGES) * FL_T * 4 + 1024;
    auto kern = k_lcp_flags<STAGES>;
    static int occ_dev[64] = {0};  // function attributes are per device: cached per device ordinal
    int dev = 0;
    cudaGetDevice(&dev);
    int& occ = occ_dev[dev & 63];
    if (!occ) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return e;
        int o = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, FL_THREADS, smem);
        if (e != cudaSuccess) return e;
        if (o < 1) return cudaErrorLaunchOutOfResources;
        occ = o;
    }
    uint64_t grid = uint64_t(sm_count) * occ;
    if (grid > p.num_tiles) grid = p.num_tiles;
    kern<<<dim3(unsigned(grid)), dim3(FL_THREADS), smem, stream>>>(tmap, p);
    return cudaGetLastError();
}

uint64_t emit_desc_words() { return uint64_t(EM_MAX_CHUNKS) * EM_DESC_WORDS; }

cudaError_t launch_emit(const EmitParams& p0, int sm_count, cudaStream_t stream) {
    EmitParams p = p0;
    static int occ_dev[64] = {0};  // function attributes are per device
    int dev = 0;
    cudaGetDevice(&dev);
    int& occ = occ_dev[dev & 63];
    if (!occ) {
        int o = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, k_cluster_emit, EM_THREADS, 0);
        if (e != cudaSuccess) return e;
        if (o < 1) return cudaErrorLaunchOutOfResources;
        occ = o;
    }
    uint64_t grid = uint64_t(sm_count) * occ;  // one chunk per CTA
    if (grid > p.num_tiles) grid = p.num_tiles;
    if (grid > EM_MAX_CHUNKS) grid = EM_MAX_CHUNKS;
    k_cluster_emit<<<dim3(unsigned(grid)), dim3(EM_THREADS), 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace e2s
