// ebwt2clust -- drop-in for the reference CLI (ref:ebwt2clust.cpp:141-198): same options, same index
// files, same X.clusters output and stdout lines; the scan itself runs on the GPU(s) through the C ABI.
// E2S_GPUS=N shards the eBWT over N GPUs of the box (contiguous ranges, host-side merge of the summaries).
#include <getopt.h>

#include <iostream>
#include <thread>

#include "host_io.hpp"

static const int min_def = 2, K_def = 16, lcp_def = 1, da_def = 4, pos_def = 1;

// the reference's help text, byte for byte (ref:ebwt2clust.cpp:34-52 as its binary prints it with the default values;
// tests/golden/help_ebwt2clust.txt is that output)
static const char* const HELP_TEXT = R"HELP(ebwt2clust [options]
Options:
-h         Print this help
-i <arg>   Input fasta file (REQUIRED)
-k <arg>   Minimum LCP required in clusters (default: 16)
-m <arg>   Discard clusters smaller than this value (default: 2)
-x <arg>   Byte size of LCP integers in input EGSA/BCR file (default: 1).
-y <arg>   Byte size of DA integers (read number) in input EGSA/BCR file (default: 4).
-z <arg>   Byte size of pos integers (position in read) in input EGSA/BCR file (default: 1).


To run ebwt2clust, you must  first build the Enhanced Generalized  Suffix Array of the input
sequences. The EGSA must be stored in the input file's folder adding extension .gesa to the
name of the input file (github.com/felipelouza/egsa), or in three files with extensions
.out, .out.lcp, .out.pairSA computed using the BCR algorithm 
(https://github.com/giovannarosone/BCR_LCP_GSA). Output is stored in reads.fasta.clusters.
)HELP";

static void help() {
    std::cout << HELP_TEXT << std::flush;
    exit(0);  // the reference exits 0 from help(), also on errors (ref:ebwt2clust.cpp:51)
}

int main(int argc, char** argv) {
    host::stamp("start");
    if (argc < 2) help();
    int k = 0, min_len = 0, lcp = 0, da = 0, pos = 0;
    std::string input;
    int opt;
    while ((opt = getopt(argc, argv, "hk:i:m:x:y:z:")) != -1) {
        switch (opt) {
            case 'h': help(); break;
            case 'k': k = atoi(optarg); break;
            case 'm': min_len = atoi(optarg); break;
            case 'i': input = optarg; break;
            case 'x': lcp = atoi(optarg); break;
            case 'y': da = atoi(optarg); break;
            case 'z': pos = atoi(optarg); break;
            default: help(); return -1;
        }
    }
    // 0 means "use the default" (ref:ebwt2clust.cpp:175-180)
    lcp = lcp == 0 ? lcp_def : lcp;
    da = da == 0 ? da_def : da;
    pos = pos == 0 ? pos_def : pos;
    k = k == 0 ? K_def : k;
    min_len = min_len == 0 ? min_def : min_len;
    if (input.empty()) help();

    host::Index idx;
    if (!idx.open(input, lcp, da, pos)) {
        std::cout << "Error: missing index files." << std::endl;  // ref:include.hpp:72-77
        return 1;
    }
    std::cout << "This is ebwt2clust. Input file: " << input << std::endl;
    host::stamp("index opened");
    auto ok = [](int v) { return v == 1 || v == 2 || v == 4 || v == 8; };
    if (!ok(lcp) || !ok(da) || !ok(pos)) {
        std::cerr << "ebwt2clust: -x/-y/-z must be 1, 2, 4 or 8" << std::endl;
        return 2;
    }
    if (idx.n < 2) {
        std::cerr << "ebwt2clust: the index holds fewer than 2 records" << std::endl;
        return 2;
    }

    // One shard per GPU (E2S_GPUS), each STREAMED through the device chunk by chunk (a chunk is a shard in time: the device holds
    // E2S_CHUNK_POSITIONS positions, default 2^28, whatever the size of the index); inputs the one-pass scan does not take
    // (an LCP value above 127, -m > 33) go through a resident shard instead.
    const std::vector<uint64_t> cuts = host::shard_cuts(idx.n, host::gpu_count_from_env());
    const int G = int(cuts.size()) - 1;
    uint64_t chunk = uint64_t(1) << 28;
    if (const char* e = getenv("E2S_CHUNK_POSITIONS"))
        if (strtoull(e, nullptr, 10)) chunk = strtoull(e, nullptr, 10);
    std::vector<e2s_ctx*> ctx(size_t(G), nullptr);
    std::vector<e2s_shard*> sh(size_t(G), nullptr);
    std::vector<e2s_cluster_summary> sums(static_cast<size_t>(G));
    std::vector<std::vector<uint8_t>> recs(static_cast<size_t>(G));  // every shard's own records, 10 bytes each, in file order
    std::vector<int> rc(size_t(G), 0);
    std::vector<std::string> errs(static_cast<size_t>(G));
    auto resident = [&](int g) -> int {  // the whole range on the device at once
        const uint64_t lo = cuts[size_t(g)], hi = cuts[size_t(g) + 1];
        if (sh[size_t(g)]) e2s_shard_destroy(sh[size_t(g)]);
        sh[size_t(g)] = nullptr;
        int r = e2s_shard_create(ctx[size_t(g)], hi - lo, lo, idx.n, &sh[size_t(g)]);
        const uint64_t a = lo >= 2 ? lo - 2 : 0, b = hi + E2S_MAX_C_LEN + 1 < idx.n ? hi + E2S_MAX_C_LEN + 1 : idx.n;
        if (!r) r = idx.load(sh[size_t(g)], a, b - a, false);
        if (!r) r = e2s_shard_set_layout(sh[size_t(g)], idx.x, idx.y, idx.z, idx.bcr ? 1 : 0);
        if (!r) r = e2s_shard_seal(sh[size_t(g)]);
        if (!r) r = e2s_cluster_run(sh[size_t(g)], uint32_t(k), min_len, &sums[size_t(g)]);
        uint64_t m = 0;
        e2s_cluster_merged none;
        memset(&none, 0, sizeof none);
        if (!r) r = e2s_cluster_finalize(sh[size_t(g)], &none);  // own records only: head / tail records are written from the merge below
        if (!r) r = e2s_cluster_count(sh[size_t(g)], &m);
        if (!r) {
            recs[size_t(g)].resize(size_t(m) * 10 + 16);
            r = e2s_cluster_fetch_packed(sh[size_t(g)], recs[size_t(g)].data(), m, &m);
            recs[size_t(g)].resize(size_t(m) * 10);
        }
        return r;
    };
    auto work = [&](int g) {
        int r = e2s_ctx_create(g, &ctx[size_t(g)]);
        if (r) { rc[size_t(g)] = r; errs[size_t(g)] = e2s_last_error(nullptr); return; }
        if (g == 0) host::stamp("context created");
        const uint64_t lo = cuts[size_t(g)], hi = cuts[size_t(g) + 1];
        bool fall_back = min_len > 33;
        if (!fall_back) {
            r = e2s_shard_create_chunked(ctx[size_t(g)], hi - lo, lo, idx.n, chunk, &sh[size_t(g)]);
            if (!r) r = e2s_shard_set_layout(sh[size_t(g)], idx.x, idx.y, idx.z, idx.bcr ? 1 : 0);
            const uint64_t cp = r ? 0 : e2s_shard_chunk_positions(sh[size_t(g)]);
            for (uint64_t clo = lo; !r && clo < hi; clo += cp) {
                const uint64_t cn = hi - clo < cp ? hi - clo : cp;
                r = e2s_chunk_begin(sh[size_t(g)], clo, cn);
                const uint64_t a = clo >= 176 ? clo - 176 : 0, b = clo + cn + E2S_MAX_C_LEN + 1 < idx.n ? clo + cn + E2S_MAX_C_LEN + 1 : idx.n;
                if (!r) r = idx.load(sh[size_t(g)], a, b - a, false);
                if (!r) r = e2s_shard_set_layout(sh[size_t(g)], idx.x, idx.y, idx.z, idx.bcr ? 1 : 0);
                uint64_t m = 0;
                if (!r) r = e2s_chunk_scan(sh[size_t(g)], uint32_t(k), min_len, 0, &m);
                if (r == E2S_ERR_UNSUPPORTED) {  // not an input for the one-pass scan, whichever chunk finds it
                    fall_back = true;
                    r = 0;
                    break;
                }
                if (!r && m) {
                    const size_t at = recs[size_t(g)].size();
                    recs[size_t(g)].resize(at + size_t(m) * 10 + 16);
                    r = e2s_cluster_fetch_packed(sh[size_t(g)], recs[size_t(g)].data() + at, m, &m);
                    recs[size_t(g)].resize(at + size_t(m) * 10);
                }
            }
            if (!r && !fall_back) r = e2s_chunked_finish(sh[size_t(g)], uint32_t(k), min_len, &sums[size_t(g)]);
        }
        if (!r && fall_back) {
            recs[size_t(g)].clear();
            r = resident(g);
        }
        if (r) { rc[size_t(g)] = r; errs[size_t(g)] = e2s_last_error(ctx[size_t(g)]); }
    };
    {
        std::vector<std::thread> th;
        for (int g = 0; g < G; ++g) th.emplace_back(work, g);
        for (auto& t : th) t.join();
    }
    host::stamp("loaded + scanned, records on the host");
    for (int g = 0; g < G; ++g)
        if (rc[size_t(g)]) {
            std::cerr << "ebwt2clust: GPU " << g << ": " << errs[size_t(g)] << std::endl;
            return 2;
        }

    FILE* out = fopen((input + ".clusters").c_str(), "wb");
    if (!out) {
        std::cerr << "ebwt2clust: cannot write " << input << ".clusters" << std::endl;
        return 2;
    }
    uint64_t n_clust_out = 0;
    auto put = [&](uint64_t st, uint64_t ln) {
        uint8_t r10[10];
        const uint16_t l16 = uint16_t(ln);
        memcpy(r10, &st, 8);
        memcpy(r10 + 8, &l16, 2);
        return fwrite(r10, 10, 1, out) == 1;
    };
    for (int g = 0; g < G; ++g) {  // every shard's slice of the file: [head record] own records [tail records]
        e2s_cluster_merged mg;
        if (e2s_cluster_merge(sums.data(), G, g, &mg)) {
            std::cerr << "ebwt2clust: " << e2s_last_error(nullptr) << std::endl;
            return 2;
        }
        bool okw = true;
        if (mg.n_prepend && mg.prepend_written) okw = put(mg.prepend_start, mg.prepend_len);
        const size_t m = recs[size_t(g)].size() / 10;
        if (okw && m) okw = fwrite(recs[size_t(g)].data(), 10, m, out) == m;
        for (uint32_t i = 0; okw && i < mg.n_append; ++i) okw = put(mg.append_start[i], mg.append_len[i]);
        if (!okw) {
            std::cerr << "ebwt2clust: short write" << std::endl;
            return 2;
        }
        n_clust_out = mg.n_clust_out;
    }
    fclose(out);
    host::stamp(".clusters written");
    // the reference counts closures in an unsigned int (ref:ebwt2clust.cpp:88,137)
    std::cout << "Done. " << static_cast<unsigned int>(n_clust_out) << " clusters saved to output file." << std::endl;
    host::quick_exit_unless_asked(0);  // (everything is on disk: skip the teardown of the CUDA contexts unless E2S_CLI_CLEAN_EXIT is set)
    for (int g = 0; g < G; ++g) {
        e2s_shard_destroy(sh[size_t(g)]);
        e2s_ctx_destroy(ctx[size_t(g)]);
    }
    host::stamp("contexts destroyed");
    return 0;
}
