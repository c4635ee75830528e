// Shards: creation (resident or chunked), the loads of the index (.gesa records, file descriptor, SoA, BCR triple, lean
// SoA), seal, and the reads staged for phase 2.

#include <stdlib.h>
#include <unistd.h>

#include <atomic>
#include <thread>

#include "host_state.h"
#include "planes.cuh"

using namespace e2s;

namespace e2s {

// every field of an index record is 1, 2, 4 or 8 bytes wide
int check_field_sizes(e2s_ctx* c, std::initializer_list<int> sizes) {
    for (int v : sizes)
        if (!(v == 1 || v == 2 || v == 4 || v == 8)) return fail(c, E2S_ERR_ARG, "field byte sizes must be 1, 2, 4 or 8");
    return E2S_OK;
}

uint64_t round_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// buf = positions the device buffers hold: the whole range (resident shard) or one chunk of it (chunked shard)
static int shard_create_impl(e2s_ctx* c, uint64_t n_local, uint64_t global_off, uint64_t n_global, uint64_t buf, e2s_shard** out) {
    if (!c || !out) return fail(c, E2S_ERR_ARG, "e2s_shard_create: NULL argument");
    *out = nullptr;
    if (n_local < 2 || global_off + n_local > n_global || (global_off != 0 && global_off < 2))
        return fail(c, E2S_ERR_ARG, "e2s_shard_create: need n_local >= 2 and a range inside [0, n_global)");
    if (n_global >= (uint64_t(1) << 47)) return fail(c, E2S_ERR_UNSUPPORTED, "e2s_shard_create: n_global must be < 2^47 positions");
    CU(c, cudaSetDevice(c->device));
    e2s_shard* s = new e2s_shard();
    s->ctx = c;
    s->n_local = n_local;
    s->global_off = global_off;
    s->n_global = n_global;
    s->alloc_r = round_up(buf, 32768) + 8192;  // whole K2 tiles (32768 positions) + one K1 tile of slack
    const size_t ne = size_t(PAD_L) + s->alloc_r;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->lcp_a), ne * 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->text_a), ne * 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->suff_a), ne * 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->bwt_a), ne);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_res), sizeof(ClusterDev));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_hist), (E2S_HIST_BINS + 1) * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_seal_flag), 4);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&s->d_planes), plane_quads(s->alloc_r) * sizeof(uint4));
    if (e != cudaSuccess) {
        e2s_shard_destroy(s);
        return fail(c, E2S_ERR_NOMEM, std::string("shard allocation: ") + cudaGetErrorString(e));
    }
    // the bit-sliced copy of the LCP the one-pass scan streams (1 B/position); without room for it the shard stays on the 4-byte stream
    if (cudaMalloc(reinterpret_cast<void**>(&s->lcpt), lcpt_bytes(s->alloc_r)) != cudaSuccess) {
        cudaGetLastError();
        s->lcpt = nullptr;
    }
    if (s->lcpt) CU(c, cudaMemsetAsync(s->lcpt, 0, lcpt_bytes(s->alloc_r), c->stream));
    CU(c, cudaMemsetAsync(s->d_planes, 0, plane_quads(s->alloc_r) * sizeof(uint4), c->stream));  // pads: code 0
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));
    s->lcp = s->lcp_a + PAD_L;
    s->text = s->text_a + PAD_L;
    s->suff = s->suff_a + PAD_L;
    s->bwt = s->bwt_a + PAD_L;
    // only the pads need defined contents (left halo of shard 0 = 0; right pad is read, never used)
    CU(c, cudaMemsetAsync(s->lcp_a, 0, PAD_L * 4, c->stream));
    CU(c, cudaMemsetAsync(s->text_a, 0, PAD_L * 4, c->stream));
    CU(c, cudaMemsetAsync(s->suff_a, 0, PAD_L * 4, c->stream));
    CU(c, cudaMemsetAsync(s->bwt_a, 0, PAD_L, c->stream));
    const size_t tail = size_t(s->alloc_r - buf);
    CU(c, cudaMemsetAsync(s->lcp + buf, 0, tail * 4, c->stream));
    CU(c, cudaMemsetAsync(s->text + buf, 0, tail * 4, c->stream));
    CU(c, cudaMemsetAsync(s->suff + buf, 0, tail * 4, c->stream));
    CU(c, cudaMemsetAsync(s->bwt + buf, 0, tail, c->stream));
    s->work = snp_work_create();
    *out = s;
    return E2S_OK;
}

// ---------------------------------------------------------------------------------------------
// chunked shards (streaming): a chunk is a shard in time
// ---------------------------------------------------------------------------------------------
// positions the buffers of a chunked shard over n_local positions hold when chunk_positions are asked for
uint64_t chunk_buffer_positions(uint64_t chunk_positions, uint64_t n_local) {
    if (chunk_positions < 16384) chunk_positions = 16384;
    chunk_positions = round_up(chunk_positions, 16384);  // chunks start at whole scan tiles
    return chunk_positions < round_up(n_local, 16384) ? chunk_positions : round_up(n_local, 16384);
}

// [first, first + count) clamped to the global range a shard keeps (2 positions of left halo, MAX_C_LEN + 1 of right halo) into
// [*a, *b); false when nothing of it is kept
static bool kept_span(const e2s_shard* s, uint64_t first, uint64_t count, uint64_t* a, uint64_t* b) {
    // (a chunk keeps PAD_L positions of left context: clusters that end in it may start up to 150 positions before it)
    const uint64_t left = s->chunked ? uint64_t(PAD_L) : 2;
    const uint64_t lo = s->global_off >= left ? s->global_off - left : 0;
    const uint64_t h = s->global_off + s->n_local + MAX_C_LEN + 1;
    const uint64_t hi = h < s->n_global ? h : s->n_global;
    *a = first > lo ? first : lo;
    *b = first + count < hi ? first + count : hi;
    return *a < *b;
}

// the two raw-record staging buffers of the loads hold at least `need` bytes each
static int ensure_raw(e2s_ctx* c, size_t need) {
    if (need <= c->raw_cap) return E2S_OK;
    CU(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 2; ++i) {
        cudaFree(c->d_raw[i]);
        c->d_raw[i] = nullptr;
    }
    c->raw_cap = 0;
    for (int i = 0; i < 2; ++i)
        if (cudaMalloc(reinterpret_cast<void**>(&c->d_raw[i]), need) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "raw staging buffer");
    c->raw_cap = need;
    return E2S_OK;
}

// the copy stream and the events every user of it shares (each is made when first missing, whichever user comes first)
int ensure_copy_stream(e2s_ctx* c) {
    if (!c->copy_stream) CU(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        if (!c->ev_copied[i]) CU(c, cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
        if (!c->ev_unpacked[i]) CU(c, cudaEventCreateWithFlags(&c->ev_unpacked[i], cudaEventDisableTiming));
    }
    if (!c->ev_start) CU(c, cudaEventCreateWithFlags(&c->ev_start, cudaEventDisableTiming));
    return E2S_OK;
}

// the scan looks at positions [-2, n_local] (on the last shard lcp[n_local] is the phantom, which only feeds END(n-1),
// left to the host tail rule): only those decide whether the byte copy is usable
static int64_t checked_hi(const e2s_shard* s) { return int64_t(s->n_local) + (s->global_off + s->n_local == s->n_global ? 0 : 1); }

// every load also writes the narrow resident copies of what it loaded (k_derive): byte LCP + base-code bit planes
static cudaError_t derive_loaded(e2s_shard* s, int64_t l, uint64_t cnt, bool have_lcp, bool have_bwt) {
    return launch_derive(s->lcp, have_bwt ? s->bwt : nullptr, have_lcp ? s->lcpt : nullptr, s->d_planes,
                         l, l + int64_t(cnt), -2, checked_hi(s), s->d_seal_flag, s->ctx->stream, s->ctx->sm_count);
}

// Called once per LCP load with the global positions [a, b) the whole call writes, before its first piece: a load over all the
// checked positions (left of global position 0 there is only the zero pad) replaces every value the last verdict came from, so
// a reloaded shard forgets it.  A partial reload keeps it (conservative: the 4-byte stream, still exact).
static cudaError_t forget_verdict_if_covered(e2s_shard* s, uint64_t a, uint64_t b) {
    const int64_t chk_lo = s->global_off >= 2 ? -2 : -int64_t(s->global_off);
    if (int64_t(a) - int64_t(s->global_off) > chk_lo || int64_t(b) - int64_t(s->global_off) < checked_hi(s)) return cudaSuccess;
    return cudaMemsetAsync(s->d_seal_flag, 0, 4, s->ctx->stream);
}

static int load_soa(e2s_shard* s, const uint32_t* lcp, const uint32_t* text, const uint32_t* suff, const uint8_t* bwt,
                    uint64_t first, uint64_t count, cudaMemcpyKind kind) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    const int64_t l = int64_t(a) - int64_t(s->global_off);
    const uint64_t so = a - first, cnt = b - a;
    if (lcp) CU(c, forget_verdict_if_covered(s, a, b));
    if (lcp) CU(c, cudaMemcpyAsync(s->lcp + l, lcp + so, cnt * 4, kind, c->stream));
    if (text) CU(c, cudaMemcpyAsync(s->text + l, text + so, cnt * 4, kind, c->stream));
    if (suff) CU(c, cudaMemcpyAsync(s->suff + l, suff + so, cnt * 4, kind, c->stream));
    if (bwt) CU(c, cudaMemcpyAsync(s->bwt + l, bwt + so, cnt, kind, c->stream));
    if (lcp || bwt) {
        CU(c, derive_loaded(s, l, cnt, lcp != nullptr, bwt != nullptr));
        ++c->launches;
    }
    s->sealed = false;
    return E2S_OK;
}

// the text / suff of the last GSA_TAIL positions of the eBWT, as far as [a, b) holds them: the phantom records past EOF are made
// of them, and clusters that start there are captured from the device
static int lean_load_tail(e2s_shard* s, uint64_t a, uint64_t b) {
    e2s_ctx* c = s->ctx;
    if (!s->host_gsa) return E2S_OK;
    const uint64_t tail_lo = s->n_global > GSA_TAIL ? s->n_global - GSA_TAIL : 0;
    const uint64_t ta = a > tail_lo ? a : tail_lo;
    if (ta >= b) return E2S_OK;
    std::vector<uint32_t> t(size_t(b - ta)), sf(size_t(b - ta));
    const int rs = s->gsa_y + s->gsa_z;
    for (uint64_t p = ta; p < b; ++p) {
        const uint8_t* g = s->host_gsa + p * uint64_t(rs);
        uint32_t vs = 0, vt = 0;
        for (int q = 0; q < (s->gsa_z < 4 ? s->gsa_z : 4); ++q) vs |= uint32_t(g[q]) << (8 * q);
        for (int q = 0; q < (s->gsa_y < 4 ? s->gsa_y : 4); ++q) vt |= uint32_t(g[s->gsa_z + q]) << (8 * q);
        sf[size_t(p - ta)] = vs;
        t[size_t(p - ta)] = vt;
    }
    const int64_t lt = int64_t(ta) - int64_t(s->global_off);
    CU(c, cudaMemcpyAsync(s->text + lt, t.data(), (b - ta) * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(s->suff + lt, sf.data(), (b - ta) * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));  // (the vectors go out of scope)
    return E2S_OK;
}

// lcp (x bytes per position) + BWT bytes of the global positions [first, first + count) -> the shard's resident arrays and their
// narrow copies.  dev: the sources are device memory (a staging buffer the caller filled), else host memory.
int load_lcp_bwt(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, uint64_t first, uint64_t count, bool dev) {
    e2s_ctx* c = s->ctx;
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_x = x;
    CU(c, forget_verdict_if_covered(s, a, b));
    const uint8_t* src = static_cast<const uint8_t*>(lcp);
    const int64_t l0 = int64_t(a) - int64_t(s->global_off);
    const cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (x == 4) {  // already at the resident width
        CU(c, cudaMemcpyAsync(s->lcp + l0, src + (a - first) * 4, (b - a) * 4, kind, c->stream));
    } else if (dev) {
        CU(c, launch_widen(src + (a - first) * uint64_t(x), x, s->lcp + l0, b - a, c->stream, c->sm_count));
        ++c->launches;
    } else {
        const uint64_t piece = uint64_t(1) << 24;
        if (int rc = ensure_raw(c, size_t(piece) * x + 64)) return rc;
        for (uint64_t p = a; p < b; p += piece) {  // (one stream: the staging buffer is free again when the widening kernel has run)
            const uint64_t cnt = b - p < piece ? b - p : piece;
            CU(c, cudaMemcpyAsync(c->d_raw[0], src + (p - first) * uint64_t(x), cnt * uint64_t(x), cudaMemcpyHostToDevice, c->stream));
            CU(c, launch_widen(c->d_raw[0], x, s->lcp + (int64_t(p) - int64_t(s->global_off)), cnt, c->stream, c->sm_count));
            ++c->launches;
        }
    }
    CU(c, cudaMemcpyAsync(s->bwt + l0, bwt + (a - first), b - a, kind, c->stream));
    CU(c, derive_loaded(s, l0, b - a, true, true));
    ++c->launches;
    s->sealed = false;
    return lean_load_tail(s, a, b);
}

// one pass over the staged reads: does any byte fall outside ACGTacgt?  (K4's consensus then needs base_to_int's general rule)
static int reads_check(e2s_ctx* c) {
    if (!c->d_reads_flag && cudaMalloc(reinterpret_cast<void**>(&c->d_reads_flag), 8) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "reads flag");
    CU(c, cudaMemsetAsync(c->d_reads_flag, 0, 8, c->stream));
    CU(c, launch_reads_check(c->d_bases, c->n_bases, c->d_off, c->n_reads, c->d_reads_flag, c->stream, c->sm_count));
    c->launches += 2;
    return E2S_OK;
}

}  // namespace e2s

extern "C" {

int e2s_shard_create(e2s_ctx* c, uint64_t n_local, uint64_t global_off, uint64_t n_global, e2s_shard** out) {
    return shard_create_impl(c, n_local, global_off, n_global, n_local, out);
}

int e2s_shard_create_chunked(e2s_ctx* c, uint64_t n_local, uint64_t global_off, uint64_t n_global, uint64_t chunk_positions,
                             e2s_shard** out) {
    const uint64_t cap = chunk_buffer_positions(chunk_positions, n_local);
    int rc = shard_create_impl(c, n_local, global_off, n_global, cap, out);
    if (rc) return rc;
    e2s_shard* s = *out;
    s->chunked = true;
    s->range_lo = global_off;
    s->range_n = n_local;
    s->chunk_cap = cap;
    memset(&s->acc, 0, sizeof s->acc);
    s->carry_state = global_off == 0 ? 0 : 1;
    if (cudaMalloc(reinterpret_cast<void**>(&s->d_cap_counters), 4 * 8) != cudaSuccess) {
        e2s_shard_destroy(s);
        *out = nullptr;
        return fail(c, E2S_ERR_NOMEM, "chunked shard counters");
    }
    CU(c, cudaMemsetAsync(s->d_cap_counters, 0, 4 * 8, c->stream));
    return E2S_OK;
}

uint64_t e2s_shard_chunk_positions(const e2s_shard* s) { return s && s->chunked ? s->chunk_cap : 0; }

// The next chunk [chunk_lo, chunk_lo + chunk_n) of the shard's range: chunks follow each other without gaps, every chunk but
// the last holds e2s_shard_chunk_positions() positions.  The loads that follow (e2s_shard_load_gesa / _soa / _soa_dev, global
// positions as always) should cover [chunk_lo - 176, chunk_lo + chunk_n + 1) as far as the eBWT reaches -- on the shard's last
// chunk + 151 as for every shard; what lies outside is ignored.
int e2s_chunk_begin(e2s_shard* s, uint64_t chunk_lo, uint64_t chunk_n) {
    if (!s || !s->chunked) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_chunk_begin: not a chunked shard");
    e2s_ctx* c = s->ctx;
    const uint64_t done = s->chunk_open || s->acc.ticket ? s->global_off + s->n_local : s->range_lo;  // (acc.ticket counts the chunks scanned)
    if (s->chunk_open) return fail(c, E2S_ERR_STATE, "e2s_chunk_begin: the previous chunk has not been scanned");
    if (chunk_lo != done || chunk_n < 1 || chunk_n > s->chunk_cap || chunk_lo + chunk_n > s->range_lo + s->range_n)
        return fail(c, E2S_ERR_ARG, "e2s_chunk_begin: chunks must follow each other and fit the buffers");
    if (chunk_lo + chunk_n < s->range_lo + s->range_n && chunk_n != s->chunk_cap)
        return fail(c, E2S_ERR_ARG, "e2s_chunk_begin: only the last chunk may be shorter than e2s_shard_chunk_positions()");
    CU(c, cudaSetDevice(c->device));
    s->global_off = chunk_lo;
    s->n_local = chunk_n;
    s->sealed = false;
    s->chunk_open = true;
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));
    if (chunk_lo < uint64_t(PAD_L)) {  // no (or a short) left context: the pad must read as zeros
        CU(c, cudaMemsetAsync(s->lcp_a, 0, PAD_L * 4, c->stream));
        CU(c, cudaMemsetAsync(s->text_a, 0, PAD_L * 4, c->stream));
        CU(c, cudaMemsetAsync(s->suff_a, 0, PAD_L * 4, c->stream));
        CU(c, cudaMemsetAsync(s->bwt_a, 0, PAD_L, c->stream));
        if (s->lcpt) CU(c, cudaMemsetAsync(s->lcpt, 0, LCPT_BLOCK, c->stream));
        CU(c, cudaMemsetAsync(s->d_planes, 0, (PL_PAD / 64) * sizeof(uint4), c->stream));
    }
    return E2S_OK;
}

void e2s_shard_destroy(e2s_shard* s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaFree(s->lcp_a);
    cudaFree(s->text_a);
    cudaFree(s->suff_a);
    cudaFree(s->bwt_a);
    cudaFree(s->lcpt);
    cudaFree(s->d_stage_dev);
    if (s->h_surv) cudaFreeHost(s->h_surv);
    if (s->h_gather) cudaFreeHost(s->h_gather);
    cudaFree(s->d_start);
    cudaFree(s->d_len);
    cudaFree(s->d_desc);
    cudaFree(s->d_row);
    cudaFree(s->d_mout);
    cudaFreeHost(s->h_mout);
    cudaFree(s->p_lcp);
    cudaFree(s->p_text);
    cudaFree(s->p_suff);
    cudaFree(s->p_bwt);
    cudaFree(s->d_surv);
    cudaFree(s->d_cap_counters);
    cudaFree(s->d_seg_start);
    cudaFree(s->d_seg_len);
    cudaFree(s->d_chunks);
    cudaFree(s->d_segs);
    cudaFree(s->d_flags);
    cudaFree(s->d_packed);
    cudaFreeHost(s->h_pin);
    cudaFree(s->d_res);
    cudaFree(s->d_hist);
    cudaFree(s->d_seal_flag);
    cudaFree(s->d_planes);
    cudaFree(s->d_pf_list);
    snp_work_destroy(s->work);
    if (s->ctx->cached == s) s->ctx->cached = nullptr;
    delete s;
}

int e2s_shard_load_gesa(e2s_shard* s, const void* records, uint64_t first, uint64_t count, int x, int y, int z) {
    if (!s || !records) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_gesa: NULL argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    CU(c, cudaSetDevice(c->device));
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = 0;
    CU(c, forget_verdict_if_covered(s, a, b));
    const int rs = x + y + z + 1;
    const uint64_t chunk = uint64_t(1) << 22;  // records per H2D chunk (multiple of 16)
    if ((rc = ensure_raw(c, size_t(chunk < (b - a) ? chunk : round_up(b - a, 16)) * rs + 64))) return rc;
    if ((rc = ensure_copy_stream(c))) return rc;
    // the copy stream starts after everything already queued on the context's stream (earlier unpack kernels read d_raw)
    CU(c, cudaEventRecord(c->ev_start, c->stream));
    CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_start, 0));
    const uint8_t* src = static_cast<const uint8_t*>(records);
    uint64_t i = 0;
    for (uint64_t p = a; p < b; p += chunk, ++i) {
        const uint64_t cnt = b - p < chunk ? b - p : chunk;
        const int buf = int(i & 1);
        if (i >= 2) CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_unpacked[buf], 0));  // the kernel that read this buffer is done
        CU(c, cudaMemcpyAsync(c->d_raw[buf], src + (p - first) * rs, size_t(cnt) * rs, cudaMemcpyHostToDevice, c->copy_stream));
        CU(c, cudaEventRecord(c->ev_copied[buf], c->copy_stream));
        CU(c, cudaStreamWaitEvent(c->stream, c->ev_copied[buf], 0));
        const int64_t l = int64_t(p) - int64_t(s->global_off);  // local index, may be -2 / -1
        CU(c, launch_unpack_gesa(c->d_raw[buf], cnt, x, y, z, s->lcp + l, s->text + l, s->suff + l, s->bwt + l, c->stream, c->sm_count));
        CU(c, cudaEventRecord(c->ev_unpacked[buf], c->stream));
        CU(c, derive_loaded(s, l, cnt, true, true));
        c->launches += 2;
    }
    s->sealed = false;
    return E2S_OK;
}

// The same straight from the file (what egsa_stream does, ref:include.hpp:42-81,120-155, instead of one istream::read per
// field): reader threads pread() pieces of the file into a ring of pinned buffers while the copy engine moves the pieces
// before them and the de-interleave kernel unpacks the ones before those.  Record i of the file = global position i.
int e2s_shard_load_gesa_fd(e2s_shard* s, int fd, uint64_t first, uint64_t count, int x, int y, int z) {
    if (!s || fd < 0) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_gesa_fd: bad argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    CU(c, cudaSetDevice(c->device));
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = 0;
    CU(c, forget_verdict_if_covered(s, a, b));
    const int rs = x + y + z + 1;
    constexpr int R = 4;                          // pinned slots
    const uint64_t piece = uint64_t(1) << 20;     // records per piece (multiple of 16)
    const size_t piece_bytes = size_t(piece) * rs + 64;
    if (c->pin_piece < piece_bytes) {
        CU(c, cudaStreamSynchronize(c->stream));
        if (c->pin_ring) cudaFreeHost(c->pin_ring);
        c->pin_ring = nullptr;
        c->pin_piece = 0;
        if (cudaHostAlloc(reinterpret_cast<void**>(&c->pin_ring), piece_bytes * R, cudaHostAllocDefault) != cudaSuccess)
            return fail(c, E2S_ERR_NOMEM, "pinned read ring");
        c->pin_piece = piece_bytes;
    }
    if ((rc = ensure_raw(c, piece_bytes))) return rc;
    if ((rc = ensure_copy_stream(c))) return rc;
    for (int i = 0; i < R; ++i)
        if (!c->ev_slot[i]) CU(c, cudaEventCreateWithFlags(&c->ev_slot[i], cudaEventDisableTiming));
    CU(c, cudaEventRecord(c->ev_start, c->stream));
    CU(c, cudaStreamWaitEvent(c->copy_stream, c->ev_start, 0));

    const uint64_t n_pieces = (b - a + piece - 1) / piece;
    std::atomic<int64_t> filled(-1), recorded(-1);  // last piece read from the file / last piece whose copy has been enqueued
    std::atomic<int> stop(0), read_err(0);
    int env_threads = 6;
    if (const char* e = getenv("E2S_READ_THREADS")) env_threads = atoi(e) > 0 ? atoi(e) : 6;
    const int T = env_threads > 16 ? 16 : env_threads;
    const int device = c->device;
    std::thread filler([&]() {
        cudaSetDevice(device);
        for (uint64_t p = 0; p < n_pieces && !stop.load(); ++p) {
            const int slot = int(p % R);
            if (p >= uint64_t(R)) {  // the copy that last read this slot must be over
                while (recorded.load(std::memory_order_acquire) < int64_t(p) - R && !stop.load()) std::this_thread::yield();
                if (stop.load()) break;
                cudaEventSynchronize(c->ev_slot[slot]);
            }
            const uint64_t p0 = a + p * piece, cnt = b - p0 < piece ? b - p0 : piece;
            uint8_t* dst = c->pin_ring + size_t(slot) * c->pin_piece;
            const size_t bytes = size_t(cnt) * rs;
            const off_t off0 = off_t(p0) * rs;
            auto part = [&](int t) {  // thread t of T: its share of the piece, 4 KB granules
                size_t lo_b = (bytes * size_t(t) / size_t(T)) & ~size_t(4095), hi_b = t + 1 == T ? bytes : (bytes * size_t(t + 1) / size_t(T)) & ~size_t(4095);
                while (lo_b < hi_b) {
                    const ssize_t got = pread(fd, dst + lo_b, hi_b - lo_b, off0 + off_t(lo_b));
                    if (got <= 0) {
                        read_err.store(1);
                        return;
                    }
                    lo_b += size_t(got);
                }
            };
            std::vector<std::thread> th;
            for (int t = 1; t < T; ++t) th.emplace_back(part, t);
            part(0);
            for (auto& w : th) w.join();
            filled.store(int64_t(p), std::memory_order_release);
            if (read_err.load()) break;
        }
    });
    rc = E2S_OK;
    cudaError_t ce = cudaSuccess;
    for (uint64_t p = 0; p < n_pieces && ce == cudaSuccess; ++p) {
        while (filled.load(std::memory_order_acquire) < int64_t(p) && !read_err.load()) std::this_thread::yield();
        if (read_err.load()) {
            rc = E2S_ERR_ARG;
            break;
        }
        const int slot = int(p % R), buf = int(p & 1);
        const uint64_t p0 = a + p * piece, cnt = b - p0 < piece ? b - p0 : piece;
        if (p >= 2) ce = cudaStreamWaitEvent(c->copy_stream, c->ev_unpacked[buf], 0);  // the kernel that read this device buffer is done
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(c->d_raw[buf], c->pin_ring + size_t(slot) * c->pin_piece, size_t(cnt) * rs, cudaMemcpyHostToDevice, c->copy_stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->ev_copied[buf], c->copy_stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->ev_slot[slot], c->copy_stream);
        recorded.store(int64_t(p), std::memory_order_release);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(c->stream, c->ev_copied[buf], 0);
        const int64_t l = int64_t(p0) - int64_t(s->global_off);  // local index, may be negative (left context)
        if (ce == cudaSuccess) ce = launch_unpack_gesa(c->d_raw[buf], cnt, x, y, z, s->lcp + l, s->text + l, s->suff + l, s->bwt + l, c->stream, c->sm_count);
        if (ce == cudaSuccess) ce = cudaEventRecord(c->ev_unpacked[buf], c->stream);
        if (ce == cudaSuccess) ce = derive_loaded(s, l, cnt, true, true);
        c->launches += 2;
    }
    stop.store(1);
    filler.join();
    // the ring is reused by the next call: its last copies must have left it
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->copy_stream);
    s->sealed = false;
    if (ce != cudaSuccess) return cuda_fail(c, ce, "e2s_shard_load_gesa_fd");
    if (rc) return fail(c, rc, "e2s_shard_load_gesa_fd: short read from the index file");
    return E2S_OK;
}

int e2s_shard_load_soa(e2s_shard* s, const uint32_t* lcp, const uint32_t* text, const uint32_t* suff, const uint8_t* bwt,
                       uint64_t first, uint64_t count) {
    return load_soa(s, lcp, text, suff, bwt, first, count, cudaMemcpyHostToDevice);
}
int e2s_shard_load_soa_dev(e2s_shard* s, const uint32_t* lcp, const uint32_t* text, const uint32_t* suff,
                           const uint8_t* bwt, uint64_t first, uint64_t count) {
    return load_soa(s, lcp, text, suff, bwt, first, count, cudaMemcpyDeviceToDevice);
}

// ---- lean SoA inputs (the BCR triple: X.out.lcp, X.out, X.out.pairSA; ref:include.hpp:157-188) -----------------------------
// Phase 1 and the prefilter need the LCP and the BWT only: 1 + x bytes per position cross PCIe instead of the 13 of an EGSA
// record.  text / suff (the pairSA file) stay on the host; the records of the ~0.1 % of the clusters that reach phase 2 are
// fetched from there when a chunk's survivors are captured.
int e2s_shard_host_gsa(e2s_shard* s, const void* pair_sa, int y, int z) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (!s->chunked) return fail(s->ctx, E2S_ERR_STATE, "e2s_shard_host_gsa: chunked shards only (the survivors' records are captured per chunk)");
    if (pair_sa)
        if (int rc = check_field_sizes(s->ctx, {y, z})) return rc;
    s->host_gsa = static_cast<const uint8_t*>(pair_sa);
    s->gsa_y = y;
    s->gsa_z = z;
    return E2S_OK;
}

// The whole BCR triple of [first, first + count): lcp + BWT as above, and X.out.pairSA (suff(z) then text(y) per position,
// ref:include.hpp:157-188) copied as it is in the file and split / widened on the device.
int e2s_shard_load_bcr(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, const void* pair_sa, int y, int z, uint64_t first,
                       uint64_t count) {
    if (!s || !lcp || !bwt || !pair_sa) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_bcr: NULL argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    CU(c, cudaSetDevice(c->device));
    if ((rc = load_lcp_bwt(s, lcp, x, bwt, first, count, false))) return rc;
    uint64_t a, b;
    if (!kept_span(s, first, count, &a, &b)) return E2S_OK;
    s->lay_y = y; s->lay_z = z; s->lay_bcr = 1;
    const int rs = y + z;
    const uint64_t piece = uint64_t(1) << 22;
    if ((rc = ensure_raw(c, size_t(piece) * size_t(rs) + 64))) return rc;
    const uint8_t* src = static_cast<const uint8_t*>(pair_sa);
    uint64_t i = 0;
    for (uint64_t p = a; p < b; p += piece, ++i) {  // (one stream: a staging buffer is free again when the kernel that read it has run)
        const uint64_t cnt = b - p < piece ? b - p : piece;
        const int64_t l = int64_t(p) - int64_t(s->global_off);
        CU(c, cudaMemcpyAsync(c->d_raw[i & 1], src + (p - first) * uint64_t(rs), cnt * uint64_t(rs), cudaMemcpyHostToDevice, c->stream));
        CU(c, launch_widen_pairs(c->d_raw[i & 1], z, y, s->suff + l, s->text + l, cnt, c->stream, c->sm_count));
        ++c->launches;
    }
    return E2S_OK;
}

int e2s_shard_load_lcp_bwt(e2s_shard* s, const void* lcp, int x, const uint8_t* bwt, uint64_t first, uint64_t count) {
    if (!s || !lcp || !bwt) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, "e2s_shard_load_lcp_bwt: NULL argument");
    e2s_ctx* c = s->ctx;
    if (int rc = check_field_sizes(c, {x})) return rc;
    CU(c, cudaSetDevice(c->device));
    return load_lcp_bwt(s, lcp, x, bwt, first, count, false);
}

int e2s_shard_set_layout(e2s_shard* s, int x, int y, int z, int bcr) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    if (int rc = check_field_sizes(s->ctx, {x, y, z})) return rc;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = bcr ? 1 : 0;
    s->sealed = false;
    return E2S_OK;
}

int e2s_shard_seal(e2s_shard* s) {
    if (!s) return fail(nullptr, E2S_ERR_ARG, "shard == NULL");
    e2s_ctx* c = s->ctx;
    CU(c, cudaSetDevice(c->device));
    if (s->global_off + s->n_local == s->n_global) {  // the records past EOF (a 1-block kernel) and their narrow copies
        CU(c, launch_fill_phantom(s->lcp, s->text, s->suff, s->bwt, s->n_local, HALO_R, s->lay_x, s->lay_y, s->lay_z,
                                  s->lay_bcr, c->stream));
        CU(c, derive_loaded(s, int64_t(s->n_local), HALO_R, true, true));
        c->launches += 2;
    }
    // The byte LCP and the bit planes were written by the loads themselves: sealing costs no pass over the data, only
    // the verdict whether every LCP value the scan looks at fits the byte copy (E2S_LCP_WIDE=1 keeps the 4-byte stream,
    // for A/B measurements and the tests)
    s->lcpt_ok = s->lcpt_sat = false;
    const char* wide = getenv("E2S_LCP_WIDE");
    if (s->lcpt && !(wide && atoi(wide) != 0)) {
        uint32_t h_flag = 1;
        CU(c, cudaMemcpyAsync(&h_flag, s->d_seal_flag, 4, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        s->lcpt_ok = true;
        s->lcpt_sat = h_flag != 0;
    }
    s->sealed = true;
    return E2S_OK;
}

int e2s_shard_lcp_bytes_resident(const e2s_shard* s) { return s ? (s->sealed && s->lcpt_ok ? 1 : 4) : 0; }

int e2s_reads_stage(e2s_ctx* c, const uint8_t* bases, const uint64_t* off, uint64_t n_reads) {
    if (!c || !bases || !off) return fail(c, E2S_ERR_ARG, "e2s_reads_stage: NULL argument");
    CU(c, cudaSetDevice(c->device));
    const uint64_t nb = off[n_reads];
    if (!c->reads_owned || nb + 16 > c->reads_cap_bases || (n_reads + 1) > c->reads_cap_off) {  // reuse the buffers when they fit
        if (c->reads_owned) {
            cudaFree(c->d_bases);
            cudaFree(c->d_off);
        }
        c->d_bases = nullptr;
        c->d_off = nullptr;
        c->reads_owned = true;
        c->reads_cap_bases = c->reads_cap_off = 0;
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&c->d_bases), nb + 16);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->d_off), (n_reads + 1) * 8);
        if (e != cudaSuccess) return fail(c, E2S_ERR_NOMEM, "reads allocation");
        c->reads_cap_bases = nb + 16;
        c->reads_cap_off = n_reads + 1;
    }
    CU(c, cudaMemcpyAsync(c->d_bases, bases, nb, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(c->d_off, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    c->n_reads = n_reads;
    c->n_bases = nb;
    return reads_check(c);
}

int e2s_reads_stage_dev(e2s_ctx* c, const uint8_t* d_bases, const uint64_t* d_off, uint64_t n_reads, uint64_t n_bases) {
    if (!c || !d_bases || !d_off) return fail(c, E2S_ERR_ARG, "e2s_reads_stage_dev: NULL argument");
    if (c->reads_owned) {
        cudaFree(c->d_bases);
        cudaFree(c->d_off);
    }
    c->reads_owned = false;
    c->reads_cap_bases = c->reads_cap_off = 0;
    c->d_bases = const_cast<uint8_t*>(d_bases);
    c->d_off = const_cast<uint64_t*>(d_off);
    c->n_reads = n_reads;
    c->n_bases = n_bases;
    return reads_check(c);
}

}  // extern "C"
