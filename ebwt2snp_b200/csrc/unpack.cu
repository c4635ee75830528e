// Staging kernels: de-interleave the on-disk array-of-structs EGSA records into the
// structure-of-arrays layout the hot kernels stream (replaces the field-by-field istream::read of
// egsa_stream::read_el, ref:include.hpp:120-199).  Reported under "staging", not under the hot path.

#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "internal.h"
#include "planes.cuh"

namespace e2s {

constexpr int UP_THREADS = 256;
constexpr int UP_RECS = 2048;  // records per tile (multiple of 16 => tile byte offset is 16B aligned)

__device__ __forceinline__ uint32_t load_le(const uint8_t* s, int nbytes) {
    uint32_t v = 0;
    const int nb = nbytes < 4 ? nbytes : 4;  // wider fields are truncated to 32 bits (ref:include.hpp:131)
    for (int b = 0; b < nb; ++b) v |= uint32_t(s[b]) << (8 * b);
    return v;
}

__global__ void __launch_bounds__(UP_THREADS) k_unpack_gesa(const uint8_t* __restrict__ rec, uint64_t count, int x, int y,
                                                            int z, uint32_t* __restrict__ lcp, uint32_t* __restrict__ text,
                                                            uint32_t* __restrict__ suff, uint8_t* __restrict__ bwt) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    const int rs = x + y + z + 1;
    const uint64_t n_tiles = (count + UP_RECS - 1) / UP_RECS;
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint64_t r0 = t * UP_RECS;
        const uint32_t nrec = uint32_t(count - r0 < UP_RECS ? count - r0 : UP_RECS);
        const uint32_t nbytes = nrec * rs;
        const uint4* src = reinterpret_cast<const uint4*>(rec + r0 * rs);  // 16B aligned: r0 % 16 == 0
        uint4* dst = reinterpret_cast<uint4*>(s_raw);
        for (uint32_t i = threadIdx.x; i < (nbytes + 15) / 16; i += UP_THREADS) dst[i] = __ldg(src + i);
        __syncthreads();
        for (uint32_t r = threadIdx.x; r < nrec; r += UP_THREADS) {
            const uint8_t* s = s_raw + r * rs;
            if (text) text[r0 + r] = load_le(s, y);
            if (suff) suff[r0 + r] = load_le(s + y, z);
            if (lcp) lcp[r0 + r] = load_le(s + y + z, x);
            if (bwt) bwt[r0 + r] = s[y + z + x];
        }
        __syncthreads();
    }
}

cudaError_t launch_unpack_gesa(const uint8_t* d_rec, uint64_t count, int x, int y, int z, uint32_t* lcp, uint32_t* text,
                               uint32_t* suff, uint8_t* bwt, cudaStream_t stream, int sm_count) {
    if (count == 0) return cudaSuccess;
    const int rs = x + y + z + 1;
    const size_t smem = size_t(UP_RECS) * rs + 16;
    cudaError_t e = cudaFuncSetAttribute(k_unpack_gesa, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    uint64_t n_tiles = (count + UP_RECS - 1) / UP_RECS;
    const uint64_t cap = uint64_t(sm_count) * 8;
    const unsigned grid = unsigned(n_tiles < cap ? n_tiles : cap);
    k_unpack_gesa<<<grid, UP_THREADS, smem, stream>>>(d_rec, count, x, y, z, lcp, text, suff, bwt);
    return cudaGetLastError();
}

// ---- the narrow resident copies, written by every load ---------------------------------------------
// The two kernels that touch every position do not need the inputs at file width (DESIGN.md section 2):
//  * the scan reads the LCP BIT-SLICED and plane-major: blocks of LCPT_BLOCK = 2048 positions, each eight runs of 32
//    64-bit words -- run p < 7 = bit plane p of the value, run 7 = the plane A, bit x = lcp[x-1] > lcp[x]; word g of a run
//    = positions 64 g .. 64 g + 63 of the block.  Values above 127 are saturated and raise *flag when they lie in the
//    range the scan looks at: the shard then stays on the 4-byte stream.  Nothing here depends on k: "lcp >= k" is a
//    7-step bit-sliced compare in the scan (scan.cu), the local-minimum test is A & ~(A >> 1);
//  * the BWT-only prefilter reads the two bit planes of the 2-bit base code.
// k_derive writes both for the local positions [a, b) that a load has just put in place -- the unpack kernel's or the
// copies' output is still in L2 -- so sealing a shard costs no pass over the data.  A load of [a, b) also refreshes bit b
// of A (its left neighbour is new), so ranges may arrive in any order.  Work unit = 16 positions; the four lanes of a
// 64-position quad combine their bits by shuffles; quads only partly inside [a, b) keep their other bits.
__device__ __forceinline__ uint32_t code_of(uint32_t c) {  // base_to_int, ref:include.hpp:265-279: ACGT/acgt -> 0..3, anything else 0
    const uint32_t u = c & 0xDFu;
    return uint32_t(u == 'C') + 2u * uint32_t(u == 'G') + 3u * uint32_t(u == 'T');
}
// bit b of the four bytes of w -> bits 0..3
__device__ __forceinline__ uint32_t gather_bit(uint32_t w, int b) { return (((w >> b) & 0x01010101u) * 0x01020408u) >> 24; }

__global__ void __launch_bounds__(256) k_derive(const uint32_t* __restrict__ lcp, const uint8_t* __restrict__ bwt,
                                                unsigned long long* __restrict__ lcpt, uint4* __restrict__ planes,
                                                int64_t a, int64_t b, int64_t chk_lo, int64_t chk_hi, uint32_t* __restrict__ flag) {
    const int64_t q_first = (a + PL_PAD) >> 6, q_last = (b + PL_PAD) >> 6;  // (position b included: its A bit)
    const int64_t n_units = (q_last - q_first + 1) * 4;
    const int lane = threadIdx.x & 31;
    uint32_t bad = 0;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t u0 = int64_t(blockIdx.x) * blockDim.x + (threadIdx.x & ~31); u0 < n_units; u0 += stride) {  // warp-uniform trip count
        const int64_t u = u0 + lane;
        const bool act = u < n_units;
        const int64_t q = q_first + (u >> 2);
        const int64_t x0 = q * 64 - PL_PAD + (u & 3) * 16;  // my 16 positions: [x0, x0 + 16)
        const int64_t lo = x0 > a ? x0 : a, hi = x0 + 16 < b ? x0 + 16 : b;
        const uint32_t cov = (act && hi > lo) ? (((1u << (hi - lo)) - 1u) << (lo - x0)) : 0u;
        // A bits: my positions in [a, b]
        const int64_t hic = x0 + 16 < b + 1 ? x0 + 16 : b + 1;
        const uint32_t covc = (act && lcpt && hic > lo) ? (((1u << (hic - lo)) - 1u) << (lo - x0)) : 0u;
        uint32_t c0 = 0, c1 = 0;
        uint32_t pl[4] = {0, 0, 0, 0};  // my 16 bits of LCP planes 2i | 2i + 1 << 16; [3] = plane 6 | A << 16
        if (cov == 0xffffu) {
            if (bwt) {
                const uint4 v = *reinterpret_cast<const uint4*>(bwt + x0);
                const uint32_t xs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const uint32_t code = code_of((xs[j >> 2] >> (8 * (j & 3))) & 0xffu);
                    c0 |= (code & 1u) << j;
                    c1 |= (code >> 1) << j;
                }
            }
            if (lcpt) {
                uint32_t prev = x0 > -int64_t(PAD_L) ? lcp[x0 - 1] : 0u;
                uint32_t abits = 0;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const uint4 v = *reinterpret_cast<const uint4*>(lcp + x0 + 4 * g);
                    const uint32_t e4[4] = {v.x, v.y, v.z, v.w};
                    uint32_t o = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int64_t x = x0 + 4 * g + j;
                        if (e4[j] > 127u && x >= chk_lo && x < chk_hi) bad = 1;
                        o |= (e4[j] > 127u ? 127u : e4[j]) << (8 * j);
                        abits |= uint32_t(prev > e4[j]) << (4 * g + j);
                        prev = e4[j];
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        pl[i] |= gather_bit(o, 2 * i) << (4 * g);
                        if (i < 3) pl[i] |= gather_bit(o, 2 * i + 1) << (16 + 4 * g);
                    }
                }
                pl[3] |= abits << 16;
            }
        } else if (cov | covc) {
            if (bwt) {
                for (int64_t x = lo; x < hi; ++x) {
                    const uint32_t code = code_of(bwt[x]);
                    c0 |= (code & 1u) << (x - x0);
                    c1 |= (code >> 1) << (x - x0);
                }
            }
            if (lcpt) {
                uint32_t prev = lo > -int64_t(PAD_L) ? lcp[lo - 1] : 0u;
                for (int64_t x = lo; x < hic; ++x) {  // (x == b: only the A bit, from whatever position b holds now)
                    const uint32_t v = lcp[x];
                    if (x < hi) {
                        if (v > 127u && x >= chk_lo && x < chk_hi) bad = 1;
                        const uint32_t vs = v > 127u ? 127u : v;
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            pl[i] |= ((vs >> (2 * i)) & 1u) << (x - x0);
                            if (i < 3) pl[i] |= ((vs >> (2 * i + 1)) & 1u) << (16 + (x - x0));
                        }
                    }
                    pl[3] |= uint32_t(prev > v) << (16 + (x - x0));
                    prev = v;
                }
            }
        }
        // the quad's four lanes -> stores by the first of them
        const int l0 = lane & ~3;
        const bool writer = act && (lane & 3) == 0;
        uint32_t cvlo = 0, cvhi = 0, cclo = 0, cchi = 0;  // coverage of the quad: positions [a, b) / [a, b]
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t cv = __shfl_sync(0xffffffffu, cov | (covc << 16), l0 + k);
            if (k < 2) {
                cvlo |= (cv & 0xffffu) << (16 * k);
                cclo |= (cv >> 16) << (16 * k);
            } else {
                cvhi |= (cv & 0xffffu) << (16 * (k - 2));
                cchi |= (cv >> 16) << (16 * (k - 2));
            }
        }
        if (planes) {  // (kernel-uniform)
            uint32_t p0lo = 0, p0hi = 0, p1lo = 0, p1hi = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t b01 = __shfl_sync(0xffffffffu, c0 | (c1 << 16), l0 + k);
                if (k < 2) {
                    p0lo |= (b01 & 0xffffu) << (16 * k);
                    p1lo |= (b01 >> 16) << (16 * k);
                } else {
                    p0hi |= (b01 & 0xffffu) << (16 * (k - 2));
                    p1hi |= (b01 >> 16) << (16 * (k - 2));
                }
            }
            if (writer && (cvlo | cvhi)) {
                uint4 o = make_uint4(p0lo, p0hi, p1lo, p1hi);
                if ((cvlo & cvhi) != 0xffffffffu) {  // partly covered: the other positions keep their bits
                    const uint4 old = planes[q];
                    o.x = (old.x & ~cvlo) | (o.x & cvlo);
                    o.y = (old.y & ~cvhi) | (o.y & cvhi);
                    o.z = (old.z & ~cvlo) | (o.z & cvlo);
                    o.w = (old.w & ~cvhi) | (o.w & cvhi);
                }
                planes[q] = o;
            }
        }
        if (lcpt) {  // (kernel-uniform) the eight words of my quad: word g of the runs of block blk
            uint32_t wlo[8] = {0, 0, 0, 0, 0, 0, 0, 0}, whi[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t v = __shfl_sync(0xffffffffu, pl[i], l0 + k);
                    if (k < 2) {
                        wlo[2 * i] |= (v & 0xffffu) << (16 * k);
                        wlo[2 * i + 1] |= (v >> 16) << (16 * k);
                    } else {
                        whi[2 * i] |= (v & 0xffffu) << (16 * (k - 2));
                        whi[2 * i + 1] |= (v >> 16) << (16 * (k - 2));
                    }
                }
            }
            const int64_t gi = q - PL_PAD / 64 + LCPT_BLOCK / 64;  // group index from the first group of the array (position -LCPT_BLOCK)
            if (writer && gi >= 0 && (cclo | cchi)) {
                unsigned long long* run0 = lcpt + (gi >> 5) * (LCPT_BLOCK / 8) + (gi & 31);
                const bool full = (cvlo & cvhi) == 0xffffffffu;  // (then [a, b] covers the quad as well)
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                    unsigned long long o = (uint64_t(whi[w]) << 32) | wlo[w];
                    if (!full) {
                        const unsigned long long m = w == 7 ? ((uint64_t(cchi) << 32) | cclo) : ((uint64_t(cvhi) << 32) | cvlo);  // run 7 = A: [a, b]
                        o = (run0[w * 32] & ~m) | (o & m);
                    }
                    run0[w * 32] = o;
                }
            }
        }
    }
    if (__syncthreads_or(int(bad)) && threadIdx.x == 0 && flag) atomicOr(flag, 1u);
}

// lcp / bwt: local position 0 of the padded arrays (a >= -PAD_L); lcpt: first byte of the bit-sliced array (the block of
// the local positions -LCPT_BLOCK .. -1).  lcpt == null: no bit-sliced LCP (bwt == null: no planes).
cudaError_t launch_derive(const uint32_t* lcp, const uint8_t* bwt, uint8_t* lcpt, uint4* planes, int64_t a, int64_t b,
                          int64_t chk_lo, int64_t chk_hi, uint32_t* flag, cudaStream_t stream, int sm_count) {
    if (b <= a || (!lcpt && !bwt)) return cudaSuccess;
    const int64_t n_units = (((b + PL_PAD) >> 6) - ((a + PL_PAD) >> 6) + 1) * 4;
    int64_t blocks = (n_units + 255) / 256;
    if (blocks > int64_t(sm_count) * 16) blocks = int64_t(sm_count) * 16;
    k_derive<<<unsigned(blocks), 256, 0, stream>>>(lcpt ? lcp : nullptr, bwt, reinterpret_cast<unsigned long long*>(lcpt),
                                                   bwt ? planes : nullptr, a, b, chk_lo, chk_hi, flag);
    return cudaGetLastError();
}

// little-endian fields of w bytes (1, 2, 4, 8) -> u32 (values wider than 32 bits truncated like the reference, ref:include.hpp:131,140,149)
__global__ void __launch_bounds__(256) k_widen(const uint8_t* __restrict__ src, int w, uint32_t* __restrict__ dst, uint64_t cnt) {
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < cnt; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint8_t* q = src + i * uint64_t(w);
        uint32_t v = q[0];
        if (w >= 2) v |= uint32_t(q[1]) << 8;
        if (w >= 4) v |= (uint32_t(q[2]) << 16) | (uint32_t(q[3]) << 24);
        dst[i] = v;
    }
}

cudaError_t launch_widen(const uint8_t* d_src, int w, uint32_t* d_dst, uint64_t cnt, cudaStream_t stream, int sm_count) {
    if (!cnt) return cudaSuccess;
    uint64_t blocks = (cnt + 255) / 256;
    if (blocks > uint64_t(sm_count) * 16) blocks = uint64_t(sm_count) * 16;
    k_widen<<<unsigned(blocks), 256, 0, stream>>>(d_src, w, d_dst, cnt);
    return cudaGetLastError();
}

// records of two little-endian fields (wa bytes, then wb bytes) -> two u32 arrays (the BCR pairSA file: suff then text)
__global__ void __launch_bounds__(256) k_widen_pairs(const uint8_t* __restrict__ src, int wa, int wb, uint32_t* __restrict__ da,
                                                     uint32_t* __restrict__ db, uint64_t cnt) {
    auto le = [](const uint8_t* q, int w) {
        uint32_t v = q[0];
        if (w >= 2) v |= uint32_t(q[1]) << 8;
        if (w >= 4) v |= (uint32_t(q[2]) << 16) | (uint32_t(q[3]) << 24);
        return v;
    };
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < cnt; i += uint64_t(gridDim.x) * blockDim.x) {
        const uint8_t* q = src + i * uint64_t(wa + wb);
        da[i] = le(q, wa);
        db[i] = le(q + wa, wb);
    }
}

cudaError_t launch_widen_pairs(const uint8_t* d_src, int wa, int wb, uint32_t* d_a, uint32_t* d_b, uint64_t cnt, cudaStream_t stream,
                               int sm_count) {
    if (!cnt) return cudaSuccess;
    uint64_t blocks = (cnt + 255) / 256;
    if (blocks > uint64_t(sm_count) * 16) blocks = uint64_t(sm_count) * 16;
    k_widen_pairs<<<unsigned(blocks), 256, 0, stream>>>(d_src, wa, wb, d_a, d_b, cnt);
    return cudaGetLastError();
}

// The record "read" after EOF (SURVEY.md 8(a) A3/B2).  read_el's temporaries share one 8-byte stack slot and a
// failed read leaves it as the last valid record left it: byte 0 = bwt[n-1] (read last); byte b >= 1 = byte b of
// the last-read field wider than b: lcp, then suff, then text for the EGSA record order (text suff lcp), lcp, then
// text, then suff for the BCR order (suff text lcp).  The phantom field of width w is the low w bytes of the slot
// (measured against the reference for ten width combinations in both formats: tests/golden, phantom_tail cases).
__global__ void k_fill_phantom(uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt, uint64_t n_local,
                               uint64_t count, int x, int y, int z, int bcr) {
    const uint8_t b0 = bwt[n_local - 1];
    const uint32_t l = lcp[n_local - 1], t = text[n_local - 1], sf = suff[n_local - 1];
    uint32_t slot = b0;  // bytes 4..7 never reach a 32-bit field
    for (int b = 1; b < 4; ++b) {
        uint32_t v = 0;
        if (b < x) v = l;
        else if (!bcr && b < z) v = sf;
        else if (b < y) v = t;
        else if (bcr && b < z) v = sf;
        slot |= v & (0xffu << (8 * b));
    }
    const uint32_t px = x >= 4 ? slot : slot & ((1u << (8 * x)) - 1u);
    const uint32_t py = y >= 4 ? slot : slot & ((1u << (8 * y)) - 1u);
    const uint32_t pz = z >= 4 ? slot : slot & ((1u << (8 * z)) - 1u);
    for (uint64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += uint64_t(gridDim.x) * blockDim.x) {
        lcp[n_local + i] = px;
        text[n_local + i] = py;
        suff[n_local + i] = pz;
        bwt[n_local + i] = b0;
    }
}

cudaError_t launch_fill_phantom(uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt, uint64_t n_local,
                                uint64_t count, int x, int y, int z, int bcr, cudaStream_t stream) {
    k_fill_phantom<<<1, 256, 0, stream>>>(lcp, text, suff, bwt, n_local, count, x, y, z, bcr);
    return cudaGetLastError();
}

}  // namespace e2s
