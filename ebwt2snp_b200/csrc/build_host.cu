// The index builder's entry points: whole index or key range, reads of one length or ragged, device or host buffers, or
// straight into a resident shard (an index larger than one call's device memory is built key range by key range).

#include <stdlib.h>

#include <functional>
#include <utility>

#include "host_state.h"

using namespace e2s;

namespace e2s {

// R + 1 HOST offsets of a ragged collection, checked as every ragged builder entry point takes them; *longest = the longest read
static int check_offsets(e2s_ctx* c, const char* who, const uint64_t* off, uint64_t n_reads, uint32_t* longest) {
    if (off[0] != 0) return fail(c, E2S_ERR_ARG, std::string(who) + ": off[0] must be 0");
    uint32_t m = 0;
    for (uint64_t r = 0; r < n_reads; ++r) {
        if (off[r + 1] < off[r]) return fail(c, E2S_ERR_ARG, std::string(who) + ": read offsets must not decrease");
        const uint64_t l = off[r + 1] - off[r];
        if (l >= 65536) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": a read of 65536 bases or more (the keys are fixed-width: short reads only)");
        m = l > m ? uint32_t(l) : m;
    }
    if (m == 0) return fail(c, E2S_ERR_ARG, std::string(who) + ": every read is empty");
    *longest = m;
    return E2S_OK;
}

// the offsets in device memory (the caller frees *d_off after synchronising the stream)
static int upload_offsets(e2s_ctx* c, const char* who, const uint64_t* off, uint64_t n_reads, uint64_t** d_off) {
    if (cudaMalloc(reinterpret_cast<void**>(d_off), (n_reads + 1) * 8) != cudaSuccess) {
        cudaGetLastError();
        *d_off = nullptr;
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": read offsets on the device");
    }
    const cudaError_t eo = cudaMemcpyAsync(*d_off, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, c->stream);
    if (eo != cudaSuccess) {
        cudaFree(*d_off);
        *d_off = nullptr;
        return cuda_fail(c, eo, "H2D read offsets");
    }
    return E2S_OK;
}

// The whole index in one call, arguments checked.  d_off == nullptr: n_reads reads of `longest` bases; else n_reads + 1 DEVICE
// offsets (off: the same in host memory), longest = the longest read.
static int build_whole(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, const uint64_t* off, uint64_t n_reads,
                       uint32_t longest, uint64_t total, uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, FieldMask mask,
                       uint64_t* ends = nullptr) {
    const cudaError_t e = build_egsa(d_reads, d_off, off, n_reads, longest, total, d_lcp, d_text, d_suff, d_bwt, c->stream, &c->launches, mask, ends);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": scratch buffers (24.5 bytes per suffix with 32-bit suffix ids, 32.5 with 64-bit ids)");
    }
    if (e == cudaErrorInvalidValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED,
                    std::string(who) + ": a read holds a base outside ACGT/acgt (N has no 2-bit code; the reference itself is "
                    "non-deterministic on N, ref:include.hpp:273) -- filter such reads first");
    }
    if (e == cudaErrorInvalidConfiguration) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": the collection is outside what one call sorts (read length < 65536, < 2^43 suffixes)");
    }
    if (e != cudaSuccess) return cuda_fail(c, e, "build_egsa");
    return E2S_OK;
}

// shared by the whole-index builder entry points of caller buffers.  off = nullptr: n_reads reads of read_len bases; else n_reads + 1
// HOST offsets.
static int build_egsa_common(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* off, uint64_t n_reads, uint32_t read_len,
                             uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt) {
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
    uint64_t total = n_reads * uint64_t(read_len);
    uint32_t longest = read_len;
    uint64_t* d_off = nullptr;
    if (off) {
        int rc = check_offsets(c, who, off, n_reads, &longest);
        if (rc == E2S_OK) rc = upload_offsets(c, who, off, n_reads, &d_off);
        if (rc != E2S_OK) return rc;
        total = off[n_reads];
    }
    const int rc = build_whole(c, who, d_reads, d_off, off, n_reads, longest, total, d_lcp, d_text, d_suff, d_bwt, FieldMask());
    if (d_off) {
        cudaStreamSynchronize(c->stream);
        cudaFree(d_off);
    }
    return rc;
}

// one key range, both read shapes (arguments checked by the caller).  d_off == nullptr: n_reads reads of read_len bases; else n_reads + 1
// DEVICE offsets, read_len = the longest read, total = off[n_reads].
static int build_range_common(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, uint64_t n_reads, uint32_t read_len,
                              uint64_t total, uint64_t key_lo, uint64_t key_hi, uint32_t before_text, uint32_t before_suff, uint64_t capacity,
                              uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position,
                              FieldMask mask = FieldMask(), uint64_t* ends = nullptr) {
    const uint64_t before = before_text == 0xffffffffu ? ~uint64_t(0) : (uint64_t(before_text) << 32) | before_suff;
    *n_records = 0;
    *first_position = 0;
    cudaError_t e = build_egsa_range(d_reads, d_off, n_reads, read_len, total, key_lo, key_hi, before, capacity, d_lcp, d_text, d_suff, d_bwt,
                                     n_records, first_position, c->stream, &c->launches, mask, ends);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": scratch buffers (24.5 / 32.5 bytes per suffix of the range)");
    }
    if (e == cudaErrorInvalidPitchValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_ARG, std::string(who) + ": the key range holds more records than `capacity` (*n_records says how many)");
    }
    if (e == cudaErrorInvalidValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": a read holds a base outside ACGT/acgt");
    }
    if (e == cudaErrorInvalidConfiguration) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": the collection is outside what one call sorts");
    }
    if (e != cudaSuccess) return cuda_fail(c, e, "build_egsa_range");
    return E2S_OK;
}

// the four index arrays of the host builder entry points on the device
struct IndexArraysDev {
    uint8_t* bwt = nullptr;
    uint32_t *lcp = nullptr, *text = nullptr, *suff = nullptr;
    // room for m positions: all four arrays or none
    cudaError_t alloc(uint64_t m) {
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&bwt), m);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&lcp), m * 4);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&text), m * 4);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&suff), m * 4);
        if (e != cudaSuccess) {
            release();
            cudaGetLastError();
        }
        return e;
    }
    void release() {
        cudaFree(bwt); cudaFree(lcp); cudaFree(text); cudaFree(suff);
        bwt = nullptr;
        lcp = text = suff = nullptr;
    }
    // the first m positions to the host arrays, then a synchronisation
    cudaError_t to_host(uint32_t* h_lcp, uint32_t* h_text, uint32_t* h_suff, uint8_t* h_bwt, uint64_t m, cudaStream_t stream) const {
        cudaError_t e = cudaMemcpyAsync(h_lcp, lcp, m * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_text, text, m * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_suff, suff, m * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_bwt, bwt, m, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        return e;
    }
};

// Where the builder puts the index: host arrays (each key range is copied there from device buffers of one range), or device
// arrays written in place (a shard's: `written` then runs on the local positions [l, l + m) just written).  Either way the arrays
// start at the index position of the first record the build writes.
struct IndexDest {
    uint32_t *lcp, *text, *suff;
    uint8_t* bwt;
    bool device;
    FieldMask mask;
    std::function<int(uint64_t l, uint64_t m)> written;
};

// The records of the key interval [lo, hi) (hi = 0: to the end of the key space) that do not fit one call's device memory (scratch
// 24.5 / 32.5 B per suffix, + 13 B of outputs when they go to the host): sub-range by sub-range (build_range_common), each one's
// records to their place in `out`.  They must be the n_range positions of the index from position at0.  d_off == nullptr: n_reads
// reads of read_len bases; else DEVICE offsets, read_len = the longest read.  A sub-range that turns out to hold more than `cap`
// records is cut in two.  ends (not null): the first and last record at full width.  E2S_ERR_ARG: the interval's records are not
// those positions.
static int build_egsa_ranges(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, uint64_t n_reads, uint32_t read_len,
                             uint64_t total, uint64_t lo0, uint64_t hi0, uint64_t at0, uint64_t n_range, uint64_t cap, const IndexDest& out,
                             uint64_t* ends) {
    const char* range_who = d_off ? "e2s_build_egsa_ragged_range_dev" : "e2s_build_egsa_range_dev";
    const uint64_t end = at0 + n_range;
    IndexArraysDev d;
    if (!out.device && d.alloc(cap) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, std::string(who) + ": device buffers of one key range");
    // sub-ranges as (lo, hi) with hi = 0 for "to the end of the key space", processed in key order from a stack
    uint64_t parts = 1;
    if (n_range > cap) {
        parts = (n_range + cap - 1) / cap;
        parts += parts / 4 + 1;
    }
    using u128 = unsigned __int128;
    const u128 width0 = (hi0 == 0 ? u128(1) << 64 : u128(hi0)) - lo0;
    std::vector<std::pair<uint64_t, uint64_t>> todo;
    for (uint64_t i = parts; i-- > 0;) {
        const uint64_t lo = lo0 + uint64_t(width0 * i / parts);
        const uint64_t hi = i + 1 == parts ? hi0 : lo0 + uint64_t(width0 * (i + 1) / parts);
        if (i + 1 == parts || hi != lo) todo.emplace_back(lo, hi);
    }
    uint64_t at = at0;
    uint64_t before = ~uint64_t(0);  // the last record so far, text << 32 | suff at full width
    int rc = E2S_OK;
    auto mismatch = [&]() {
        return fail(c, E2S_ERR_ARG, std::string(who) + ": the key range's records are not index positions [" + std::to_string(at0) + ", " +
                                        std::to_string(end) + ")");
    };
    while (!todo.empty() && rc == E2S_OK) {
        const auto [lo, hi] = todo.back();
        todo.pop_back();
        uint64_t m = 0, first = 0, got[2] = {before, before};
        // (in place: a range never writes past the end of the arrays)
        const uint64_t room = out.device && end - at < cap ? end - at : cap;
        const uint64_t l = at - at0;
        rc = build_range_common(c, range_who, d_reads, d_off, n_reads, read_len, total, lo, hi, uint32_t(before >> 32), uint32_t(before), room,
                                out.device ? out.lcp + l : d.lcp, out.device ? out.text + l : d.text, out.device ? out.suff + l : d.suff,
                                out.device ? out.bwt + l : d.bwt, &m, &first, out.mask, got);
        if (rc == E2S_ERR_ARG && m > room) {  // too many records for the buffers: two halves (a single key value cannot be cut)
            if (m > end - at) {
                rc = mismatch();
                break;
            }
            const u128 width = (hi == 0 ? u128(1) << 64 : u128(hi)) - lo;
            if (width == 1) {
                rc = fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": one 32-symbol prefix is shared by more suffixes than fit the device");
                break;
            }
            const uint64_t mid = lo + uint64_t(width >> 1);
            todo.emplace_back(mid, hi);
            todo.emplace_back(lo, mid);
            rc = E2S_OK;
            continue;
        }
        if (rc != E2S_OK) break;
        if (first != at || m > end - at) {
            rc = mismatch();
            break;
        }
        if (m) {
            if (out.device) {
                rc = out.written(l, m);
            } else {
                const cudaError_t e = d.to_host(out.lcp + l, out.text + l, out.suff + l, out.bwt + l, m, c->stream);
                if (e != cudaSuccess) rc = cuda_fail(c, e, "D2H index arrays of a key range");
            }
            if (ends && at == at0) ends[0] = got[0];
            at += m;
            before = got[1];
        }
    }
    if (rc == E2S_OK && at != end) rc = mismatch();
    if (rc == E2S_OK && ends) ends[1] = before;
    d.release();
    return rc;
}

// Do the n_sort suffixes of the index of `total` bases in n_reads reads (the longest: `longest` bases) -- all of them, or one shard's
// key range -- fit one call on the device as it is now, the reads already resident?  *cap = 0: build them in one call; else the
// records per key range.  Scratch: 24.5 B per suffix sorted with 32-bit suffix ids, 32.5 with 64-bit ids (equal lengths: n < 2^32;
// ragged: R << shift, shift = the bits of the longest read's length + 1), plus out_bytes per suffix when the outputs are device buffers
// of the call; packed reads and slack (half a byte per base), and for ragged reads the 2 extra packed words and the device offset of
// every read.  0.92 of the free memory may be used.  E2S_BUILD_RANGE_RECORDS=<cap> forces key ranges (tests).
static int range_records(e2s_ctx* c, const char* who, uint64_t total, uint64_t n_reads, uint64_t n_sort, bool ragged, uint32_t longest,
                         uint64_t out_bytes, const char* advice, uint64_t* cap) {
    const uint64_t n = total + n_reads;
    bool ids64 = n > 0xffffffffull;
    if (ragged) {
        uint32_t bits = 1;
        while ((longest >> bits) != 0) ++bits;
        ids64 = n_reads > (uint64_t(1) << (32 - bits));
    }
    if (getenv("E2S_BUILD_IDS64")) ids64 = true;
    *cap = 0;
    if (const char* f = getenv("E2S_BUILD_RANGE_RECORDS")) {
        *cap = strtoull(f, nullptr, 10);
        return E2S_OK;
    }
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const uint64_t per_suffix = out_bytes + (ids64 ? 33 : 25);
    const double fixed = double(total) / 2 + (ragged ? 24.0 * double(n_reads) : 0.0);
    if (double(n_sort) * double(per_suffix) + fixed <= 0.92 * double(free_b)) return E2S_OK;
    const double room = 0.92 * double(free_b) - fixed - double(n) / 512;
    *cap = room > 0 ? uint64_t(room / double(per_suffix)) : 0;
    if (*cap < 4096) return fail(c, E2S_ERR_NOMEM, std::string(who) + ": not even one key range of the index fits the device" + advice);
    return E2S_OK;
}

// host buffers in and out: device buffers allocated and released here
static int build_egsa_host(e2s_ctx* c, const char* who, const uint8_t* reads, const uint64_t* off, uint64_t n_reads, uint32_t read_len,
                           uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt) {
    CU(c, cudaSetDevice(c->device));
    const uint64_t total = off ? off[n_reads] : n_reads * uint64_t(read_len);
    const uint64_t n = total + n_reads;
    uint32_t longest = read_len;
    if (off) {
        if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
        const int rc = check_offsets(c, who, off, n_reads, &longest);
        if (rc != E2S_OK) return rc;
    }
    uint8_t* d_reads = nullptr;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d_reads), total ? total : 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": the reads on the device");
    }
    uint64_t cap = 0;
    if (int rc = range_records(c, who, total, n_reads, n, off != nullptr, longest, 13, "", &cap)) {
        cudaFree(d_reads);
        return rc;
    }
    if (cap) {
        uint64_t* d_off = nullptr;
        int rc = E2S_OK;
        if (off) rc = upload_offsets(c, who, off, n_reads, &d_off);
        if (rc == E2S_OK) {
            e = cudaMemcpyAsync(d_reads, reads, total, cudaMemcpyHostToDevice, c->stream);
            rc = e == cudaSuccess ? build_egsa_ranges(c, who, d_reads, d_off, n_reads, longest, total, 0, 0, 0, n, cap,
                                                      IndexDest{lcp, text, suff, bwt, false, FieldMask(), nullptr}, nullptr)
                                  : cuda_fail(c, e, "H2D reads");
        }
        cudaStreamSynchronize(c->stream);
        cudaFree(d_off);
        cudaFree(d_reads);
        return rc;
    }
    IndexArraysDev d;
    if (d.alloc(n) != cudaSuccess) {
        cudaFree(d_reads);
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": device buffers");
    }
    e = cudaMemcpyAsync(d_reads, reads, total, cudaMemcpyHostToDevice, c->stream);
    int rc = e == cudaSuccess ? build_egsa_common(c, who, d_reads, off, n_reads, read_len, d.lcp, d.text, d.suff, d.bwt) : cuda_fail(c, e, "H2D reads");
    if (rc == E2S_OK && (e = d.to_host(lcp, text, suff, bwt, n, c->stream)) != cudaSuccess) rc = cuda_fail(c, e, "D2H index arrays");
    cudaFree(d_reads);
    d.release();
    return rc;
}

}  // namespace e2s

extern "C" {

int e2s_build_egsa_dev(e2s_ctx* c, const uint8_t* d_reads, uint64_t n_reads, uint32_t read_len, uint32_t* d_lcp, uint32_t* d_text,
                       uint32_t* d_suff, uint8_t* d_bwt) {
    if (!c || !d_reads || !d_lcp || !d_text || !d_suff || !d_bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_dev: NULL argument");
    if (n_reads == 0 || read_len == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_dev: empty read collection");
    CU(c, cudaSetDevice(c->device));
    return build_egsa_common(c, "e2s_build_egsa_dev", d_reads, nullptr, n_reads, read_len, d_lcp, d_text, d_suff, d_bwt);
}

int e2s_build_egsa_ragged_dev(e2s_ctx* c, const uint8_t* d_bases, const uint64_t* off, uint64_t n_reads, uint32_t* d_lcp, uint32_t* d_text,
                              uint32_t* d_suff, uint8_t* d_bwt) {
    if (!c || !d_bases || !off || !d_lcp || !d_text || !d_suff || !d_bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged_dev: NULL argument");
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged_dev: empty read collection");
    CU(c, cudaSetDevice(c->device));
    return build_egsa_common(c, "e2s_build_egsa_ragged_dev", d_bases, off, n_reads, 0, d_lcp, d_text, d_suff, d_bwt);
}

int e2s_build_egsa_range_dev(e2s_ctx* c, const uint8_t* d_reads, uint64_t n_reads, uint32_t read_len, uint64_t key_lo, uint64_t key_hi,
                             uint32_t before_text, uint32_t before_suff, uint64_t capacity, uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff,
                             uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position) {
    if (!c || !d_reads || !d_lcp || !d_text || !d_suff || !d_bwt || !n_records || !first_position)
        return fail(c, E2S_ERR_ARG, "e2s_build_egsa_range_dev: NULL argument");
    if (n_reads == 0 || read_len == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_range_dev: empty read collection");
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, "e2s_build_egsa_range_dev: more than 2^32 - 1 reads (text is a 32-bit field)");
    if (key_hi != 0 && key_hi <= key_lo) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_range_dev: empty key range");
    CU(c, cudaSetDevice(c->device));
    return build_range_common(c, "e2s_build_egsa_range_dev", d_reads, nullptr, n_reads, read_len, n_reads * uint64_t(read_len), key_lo, key_hi,
                              before_text, before_suff, capacity, d_lcp, d_text, d_suff, d_bwt, n_records, first_position);
}

int e2s_build_egsa_ragged_range_dev(e2s_ctx* c, const uint8_t* d_bases, const uint64_t* off, uint64_t n_reads, uint64_t key_lo, uint64_t key_hi,
                                    uint32_t before_text, uint32_t before_suff, uint64_t capacity, uint32_t* d_lcp, uint32_t* d_text,
                                    uint32_t* d_suff, uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position) {
    const char* who = "e2s_build_egsa_ragged_range_dev";
    if (!c || !d_bases || !off || !d_lcp || !d_text || !d_suff || !d_bwt || !n_records || !first_position)
        return fail(c, E2S_ERR_ARG, std::string(who) + ": NULL argument");
    *n_records = 0;
    *first_position = 0;
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, std::string(who) + ": empty read collection");
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
    if (key_hi != 0 && key_hi <= key_lo) return fail(c, E2S_ERR_ARG, std::string(who) + ": empty key range");
    CU(c, cudaSetDevice(c->device));
    uint32_t longest = 0;
    uint64_t* d_off = nullptr;
    int rc = check_offsets(c, who, off, n_reads, &longest);
    if (rc == E2S_OK) rc = upload_offsets(c, who, off, n_reads, &d_off);
    if (rc != E2S_OK) return rc;
    rc = build_range_common(c, who, d_bases, d_off, n_reads, longest, off[n_reads], key_lo, key_hi, before_text, before_suff, capacity, d_lcp, d_text,
                            d_suff, d_bwt, n_records, first_position);
    cudaStreamSynchronize(c->stream);
    cudaFree(d_off);
    return rc;
}

int e2s_build_egsa(e2s_ctx* c, const uint8_t* reads, uint64_t n_reads, uint32_t read_len, uint32_t* lcp, uint32_t* text, uint32_t* suff,
                   uint8_t* bwt) {
    if (!c || !reads || !lcp || !text || !suff || !bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa: NULL argument");
    if (n_reads == 0 || read_len == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa: empty read collection");
    return build_egsa_host(c, "e2s_build_egsa", reads, nullptr, n_reads, read_len, lcp, text, suff, bwt);
}

int e2s_build_egsa_ragged(e2s_ctx* c, const uint8_t* bases, const uint64_t* off, uint64_t n_reads, uint32_t* lcp, uint32_t* text,
                          uint32_t* suff, uint8_t* bwt) {
    if (!c || !bases || !off || !lcp || !text || !suff || !bwt) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged: NULL argument");
    if (n_reads == 0) return fail(c, E2S_ERR_ARG, "e2s_build_egsa_ragged: empty read collection");
    return build_egsa_host(c, "e2s_build_egsa_ragged", bases, off, n_reads, 0, lcp, text, suff, bwt);
}

// The records of the key range [key_lo, key_hi) of the staged reads' index written straight into a resident shard's arrays, each field
// kept at its .gesa width, then the narrow copies of what was written.  The staged reads (and, for ragged reads, their staged device
// offsets) are the builder's input.  The whole key space (0, 0) on a shard of the whole index is one build when its scratch fits.
int e2s_shard_build_egsa_range(e2s_shard* s, const uint64_t* off, uint64_t key_lo, uint64_t key_hi, int x, int y, int z) {
    const char* who = "e2s_shard_build_egsa";
    if (!s || !off) return fail(s ? s->ctx : nullptr, E2S_ERR_ARG, std::string(who) + ": NULL argument");
    e2s_ctx* c = s->ctx;
    int rc;
    if ((rc = check_field_sizes(c, {x, y, z}))) return rc;
    if (s->chunked) return fail(c, E2S_ERR_ARG, std::string(who) + ": needs a resident shard (not chunked)");
    if (key_hi != 0 && key_hi <= key_lo) return fail(c, E2S_ERR_ARG, std::string(who) + ": empty key range");
    if (!c->d_bases || !c->d_off || c->n_reads == 0) return fail(c, E2S_ERR_STATE, std::string(who) + ": stage the reads first (e2s_reads_stage)");
    const uint64_t n_reads = c->n_reads;
    if (off[n_reads] != c->n_bases) return fail(c, E2S_ERR_ARG, std::string(who) + ": `off` does not describe the staged reads");
    if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
    uint32_t longest = 0;
    if ((rc = check_offsets(c, who, off, n_reads, &longest))) return rc;
    const uint64_t total = off[n_reads], n = total + n_reads;
    if (s->n_global != n) return fail(c, E2S_ERR_ARG, std::string(who) + ": the shard's n_global must be off[n_reads] + n_reads");
    const bool whole = key_lo == 0 && key_hi == 0;
    if (whole && s->n_local != n) return fail(c, E2S_ERR_ARG, std::string(who) + ": the whole key space needs a shard of the whole eBWT");
    const bool ragged = total != n_reads * uint64_t(longest);  // (every read has `longest` bases exactly when the sum says so)
    CU(c, cudaSetDevice(c->device));
    uint64_t cap = 0;
    if ((rc = range_records(c, who, total, n_reads, s->n_local, ragged, longest, 0,
                            " next to the shard; split the index over more shards, or build the index file with build_gesa and stream "
                            "it (ebwt2clust / clust2snp, e2s_pipeline_host)",
                            &cap)))
        return rc;
    auto mask = [](int w) { return w >= 4 ? ~0u : (1u << (8 * w)) - 1u; };
    const FieldMask fm{mask(x), mask(y), mask(z)};
    auto written = [&](uint64_t l, uint64_t m) -> int {
        CU(c, derive_loaded(s, int64_t(l), m, true, true));
        ++c->launches;
        return E2S_OK;
    };
    s->sealed = false;
    s->ends_known = false;
    s->lay_x = x; s->lay_y = y; s->lay_z = z; s->lay_bcr = 0;
    CU(c, cudaMemsetAsync(s->d_seal_flag, 0, 4, c->stream));  // every position is rewritten: the old verdict goes
    const uint64_t* d_off = ragged ? c->d_off : nullptr;
    if (whole && !cap) {
        if ((rc = build_whole(c, who, c->d_bases, d_off, off, n_reads, longest, total, s->lcp, s->text, s->suff, s->bwt, fm, s->ends))) return rc;
        rc = written(0, n);
    } else {
        rc = build_egsa_ranges(c, who, c->d_bases, d_off, n_reads, longest, total, key_lo, key_hi, s->global_off, s->n_local, cap ? cap : s->n_local,
                               IndexDest{s->lcp, s->text, s->suff, s->bwt, true, fm, written}, s->ends);
    }
    s->ends_known = rc == E2S_OK;
    return rc;
}

int e2s_shard_build_egsa(e2s_shard* s, const uint64_t* off, int x, int y, int z) { return e2s_shard_build_egsa_range(s, off, 0, 0, x, y, z); }

// Cuts of the key space into `parts` shards of the staged reads' index (the builder's key words and slot map, a fixed-stride sample).
int e2s_reads_key_cuts(e2s_ctx* c, const uint64_t* off, int parts, uint64_t* key_lo, uint64_t* position) {
    const char* who = "e2s_reads_key_cuts";
    if (!c || !off || !key_lo || !position) return fail(c, E2S_ERR_ARG, std::string(who) + ": NULL argument");
    if (parts < 1) return fail(c, E2S_ERR_ARG, std::string(who) + ": parts must be at least 1");
    if (!c->d_bases || !c->d_off || c->n_reads == 0) return fail(c, E2S_ERR_STATE, std::string(who) + ": stage the reads first (e2s_reads_stage)");
    const uint64_t n_reads = c->n_reads;
    if (off[n_reads] != c->n_bases) return fail(c, E2S_ERR_ARG, std::string(who) + ": `off` does not describe the staged reads");
    uint32_t longest = 0;
    int rc;
    if ((rc = check_offsets(c, who, off, n_reads, &longest))) return rc;
    const uint64_t total = off[n_reads], n = total + n_reads;
    if (uint64_t(parts) * 2 > n) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": too many shards for this collection (each needs 2 positions)");
    if (parts > 1024) return fail(c, E2S_ERR_ARG, std::string(who) + ": at most 1024 parts");
    if (parts == 1) {  // the whole key space: nothing to sample or count
        key_lo[0] = 0;
        position[0] = 0;
        position[1] = n;
        return E2S_OK;
    }
    const bool ragged = total != n_reads * uint64_t(longest);
    CU(c, cudaSetDevice(c->device));
    const cudaError_t e = key_cuts(c->d_bases, ragged ? c->d_off : nullptr, n_reads, longest, total, uint32_t(parts), key_lo, position, c->stream,
                                   &c->launches);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": the packed reads (a quarter byte per base)");
    }
    if (e == cudaErrorInvalidValue) {
        cudaGetLastError();
        return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": a read holds a base outside ACGT/acgt");
    }
    if (e != cudaErrorInvalidConfiguration && e != cudaSuccess) return cuda_fail(c, e, "key_cuts");
    for (int i = 0; i < parts && e == cudaSuccess; ++i)
        if (position[i + 1] - position[i] < 2) {
            return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": too many shards for this collection (a key range holds fewer than 2 "
                                                                   "positions; one key value cannot be split)");
        }
    if (e != cudaSuccess) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": too many shards for this collection (the cuts cannot increase)");
    return E2S_OK;
}

}  // extern "C"
