// The index builder's entry points: whole index or key range, reads of one length or ragged, device or host buffers
// (a host index larger than one call's device memory is built key range by key range).

#include <stdlib.h>

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

// shared by the four whole-index builder entry points.  off = nullptr: n_reads reads of read_len bases; else n_reads + 1 HOST offsets.
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
    cudaError_t e = build_egsa(d_reads, d_off, off, n_reads, longest, total, d_lcp, d_text, d_suff, d_bwt, c->stream, &c->launches);
    if (d_off) {
        cudaStreamSynchronize(c->stream);
        cudaFree(d_off);
    }
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

// one key range, both read shapes (arguments checked by the caller).  d_off == nullptr: n_reads reads of read_len bases; else n_reads + 1
// DEVICE offsets, read_len = the longest read, total = off[n_reads].
static int build_range_common(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, uint64_t n_reads, uint32_t read_len,
                              uint64_t total, uint64_t key_lo, uint64_t key_hi, uint32_t before_text, uint32_t before_suff, uint64_t capacity,
                              uint32_t* d_lcp, uint32_t* d_text, uint32_t* d_suff, uint8_t* d_bwt, uint64_t* n_records, uint64_t* first_position) {
    const uint64_t before = before_text == 0xffffffffu ? ~uint64_t(0) : (uint64_t(before_text) << 32) | before_suff;
    *n_records = 0;
    *first_position = 0;
    cudaError_t e = build_egsa_range(d_reads, d_off, n_reads, read_len, total, key_lo, key_hi, before, capacity, d_lcp, d_text, d_suff, d_bwt,
                                     n_records, first_position, c->stream, &c->launches);
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

// An index that does not fit one call's device memory (outputs 13 B + scratch 24.5 / 32.5 B per suffix): the index key range by key
// range (build_range_common), every range's records copied to their place in the host arrays.  d_off == nullptr: n_reads reads of
// read_len bases; else DEVICE offsets (uploaded once for all ranges), read_len = the longest read.  A range that turns out to hold more
// than `cap` records is cut in two.  E2S_BUILD_RANGE_RECORDS=<cap> forces this path (tests).
static int build_egsa_host_ranges(e2s_ctx* c, const char* who, const uint8_t* d_reads, const uint64_t* d_off, uint64_t n_reads, uint32_t read_len,
                                  uint64_t total, uint64_t cap, uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt) {
    const char* range_who = d_off ? "e2s_build_egsa_ragged_range_dev" : "e2s_build_egsa_range_dev";
    const uint64_t n = total + n_reads;
    IndexArraysDev d;
    if (d.alloc(cap) != cudaSuccess) return fail(c, E2S_ERR_NOMEM, std::string(who) + ": device buffers of one key range");
    // ranges as (lo, hi) with hi = 0 for "to the end of the key space", processed in key order from a stack
    uint64_t parts = (n + cap - 1) / cap;
    parts += parts / 4 + 1;
    std::vector<std::pair<uint64_t, uint64_t>> todo;
    for (uint64_t i = parts; i-- > 0;) {
        const uint64_t lo = uint64_t((static_cast<unsigned __int128>(i) << 64) / parts);
        const uint64_t hi = i + 1 == parts ? 0 : uint64_t((static_cast<unsigned __int128>(i + 1) << 64) / parts);
        if (hi == 0 || hi > lo) todo.emplace_back(lo, hi);
    }
    uint64_t at = 0;
    uint32_t before_text = 0xffffffffu, before_suff = 0;
    int rc = E2S_OK;
    while (!todo.empty() && rc == E2S_OK) {
        const auto [lo, hi] = todo.back();
        todo.pop_back();
        uint64_t m = 0, first = 0;
        rc = build_range_common(c, range_who, d_reads, d_off, n_reads, read_len, total, lo, hi, before_text, before_suff, cap, d.lcp, d.text, d.suff,
                                d.bwt, &m, &first);
        if (rc == E2S_ERR_ARG && m > cap) {  // too many records for the buffers: two halves (a single key value cannot be cut)
            const uint64_t width = hi - lo;  // (mod 2^64: right for hi = 0 as long as lo > 0 or the range is not the whole space)
            if (width == 1 || (lo == 0 && hi == 0)) {
                rc = fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": one 32-symbol prefix is shared by more suffixes than fit the device");
                break;
            }
            const uint64_t mid = lo + (width >> 1);
            todo.emplace_back(mid, hi);
            todo.emplace_back(lo, mid);
            rc = E2S_OK;
            continue;
        }
        if (rc != E2S_OK) break;
        if (first != at || at + m > n) {
            rc = fail(c, E2S_ERR_STATE, std::string(who) + ": key ranges do not tile the index");
            break;
        }
        if (m) {
            const cudaError_t e = d.to_host(lcp + at, text + at, suff + at, bwt + at, m, c->stream);
            if (e != cudaSuccess) {
                rc = cuda_fail(c, e, "D2H index arrays of a key range");
                break;
            }
            at += m;
            before_text = text[at - 1];
            before_suff = suff[at - 1];
        }
    }
    if (rc == E2S_OK && at != n) rc = fail(c, E2S_ERR_STATE, std::string(who) + ": key ranges do not cover the index");
    d.release();
    return rc;
}

// host buffers in and out: device buffers allocated and released here
static int build_egsa_host(e2s_ctx* c, const char* who, const uint8_t* reads, const uint64_t* off, uint64_t n_reads, uint32_t read_len,
                           uint32_t* lcp, uint32_t* text, uint32_t* suff, uint8_t* bwt) {
    CU(c, cudaSetDevice(c->device));
    const uint64_t total = off ? off[n_reads] : n_reads * uint64_t(read_len);
    const uint64_t n = total + n_reads;
    // suffix ids are 64-bit beyond 2^32 (equal lengths: n; ragged: R << shift, shift = the bits of the longest read's length + 1)
    bool ids64 = n > 0xffffffffull;
    uint32_t longest = read_len;
    if (off) {
        if (n_reads > 0xffffffffull) return fail(c, E2S_ERR_UNSUPPORTED, std::string(who) + ": more than 2^32 - 1 reads (text is a 32-bit field)");
        const int rc = check_offsets(c, who, off, n_reads, &longest);
        if (rc != E2S_OK) return rc;
        uint32_t bits = 1;
        while ((longest >> bits) != 0) ++bits;
        ids64 = n_reads > (uint64_t(1) << (32 - bits));
    }
    if (getenv("E2S_BUILD_IDS64")) ids64 = true;
    uint8_t* d_reads = nullptr;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d_reads), total ? total : 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(c, E2S_ERR_NOMEM, std::string(who) + ": the reads on the device");
    }
    {   // does the whole index fit one call?  13 B of outputs + up to 32.5 B of scratch per suffix, packed reads and slack (half a byte
        // per base), and for ragged reads the 2 extra packed words and the device offset of every read; the reads are already resident
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const uint64_t per_suffix = 13 + (ids64 ? 33 : 25);
        const double fixed = double(total) / 2 + (off ? 24.0 * double(n_reads) : 0.0);
        uint64_t cap = 0;
        if (const char* f = getenv("E2S_BUILD_RANGE_RECORDS")) cap = strtoull(f, nullptr, 10);
        else if (double(n) * double(per_suffix) + fixed > 0.92 * double(free_b)) {
            const double room = 0.92 * double(free_b) - fixed - double(n) / 512;
            cap = room > 0 ? uint64_t(room / double(per_suffix)) : 0;
            if (cap < 4096) {
                cudaFree(d_reads);
                return fail(c, E2S_ERR_NOMEM, std::string(who) + ": not even one key range of the index fits the device");
            }
        }
        if (cap) {
            uint64_t* d_off = nullptr;
            int rc = E2S_OK;
            if (off) rc = upload_offsets(c, who, off, n_reads, &d_off);
            if (rc == E2S_OK) {
                e = cudaMemcpyAsync(d_reads, reads, total, cudaMemcpyHostToDevice, c->stream);
                rc = e == cudaSuccess ? build_egsa_host_ranges(c, who, d_reads, d_off, n_reads, longest, total, cap, lcp, text, suff, bwt)
                                      : cuda_fail(c, e, "H2D reads");
            }
            cudaStreamSynchronize(c->stream);
            cudaFree(d_off);
            cudaFree(d_reads);
            return rc;
        }
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

}  // extern "C"
