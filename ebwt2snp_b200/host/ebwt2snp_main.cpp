// ebwt2snp -- reads to SNPs in one process and one CUDA context: the FASTA's reads cross PCIe once, the index is built on the
// GPU straight into the resident shard that scans it (no X.gesa), then ebwt2clust and clust2snp run on that shard.  Writes the
// X.clusters and the .snp file that `build_gesa -x -y -z`, `ebwt2clust` and `clust2snp` with the same options write, and prints
// the counting lines of both tools.  The calls are those of e2s_pipeline_reads, made one by one so that the records and events
// are fetched at the sizes the step reports.  -G 1 (the default): one GPU, the whole eBWT and the reads must fit it.  -G N: the
// index is split into N shards by key range, each built from the reads on its GPU (shard g on device g % devices), then the
// multi-shard sequence of ebwt2clust runs over them; the files are the same.
#include <getopt.h>

#include <functional>
#include <iostream>
#include <thread>

#include "host_io.hpp"

static void help() {
    std::cout << "ebwt2snp [options]\nOptions:\n"
                 "-h          Print this help.\n"
                 "-i <arg>    Input fasta file containing the samples' reads (REQUIRED). Outputs: <arg>.clusters and the .snp\n"
                 "            file clust2snp writes for it.\n"
                 "-n <arg>    Number of reads in the first sample (REQUIRED).\n"
                 "-k <arg>    Minimum LCP required in clusters (ebwt2clust -k; default: 16).\n"
                 "-l <arg>    Discard clusters smaller than this value (ebwt2clust -m; default: 2).\n"
                 "-L <arg>    Length of left-context, SNP included (default: 31).\n"
                 "-R <arg>    Length of right context, SNP excluded (default: 30).\n"
                 "-g <arg>    Maximum allowed gap length in indel (default: 10). If 0, indels are disabled.\n"
                 "-v <arg>    Maximum number of non-isolated SNPs in left-contexts (default: 3).\n"
                 "-c <arg>    Extract this maximum number of reads per individual to compute consensus of left-context (default: 20).\n"
                 "-e <arg>    Mismatches allowed between DNA fragments forming consensus of left-context (default: 2).\n"
                 "-m <arg>    Minimum cluster length per individual (clust2snp -m; default: 5).\n"
                 "-p <arg>    Automatically choose max cluster length so that this fraction of bases is analyzed (default: 0.99).\n"
                 "-x <arg>    Byte size of LCP integers of the index, as build_gesa -x would write them (default: 1).\n"
                 "-y <arg>    Byte size of DA integers (read number) (default: 4).\n"
                 "-z <arg>    Byte size of pos integers (position in read) (default: 1).\n"
                 "-G <arg>    Number of shards the index is split over, by key range (default: 1). Shard g is built and kept\n"
                 "            on GPU g % (GPUs visible); shards that share a GPU run one after another. Same output files.\n"
                 "\n"
                 "Builds the index on the GPU(s) and keeps it there: no index file is written or read. The GPUs come from -G\n"
                 "alone (E2S_GPUS is\n"
                 "ignored); a shard takes 14.25 bytes per position on its device, and every device holds all the reads. For an\n"
                 "index larger than the GPUs, reads containing N or the BCR (-b) layout, run build_gesa, ebwt2clust and\n"
                 "clust2snp.\n"
              << std::flush;
    exit(0);
}

// the .snp next to the FASTA, as clust2snp names it; 3 when there is no candidate (clust2snp writes no .snp then either)
static int write_snp(const std::string& input, const std::vector<e2s_event>& ev, const e2s_snp_params& p, uint64_t n_candidates, bool saw_n) {
    std::cout << "Done. " << n_candidates << " potential variants detected (some might be detected twice: on fw and rev strands)" << std::endl;
    if (saw_n)
        std::cerr << "ebwt2snp: warning: N bases met; the reference maps them through rand() (ref:include.hpp:273), here they count as A" << std::endl;
    if (n_candidates == 0) {
        std::cerr << "ebwt2snp: no candidate variants; no .snp written" << std::endl;
        return 3;
    }
    char* text = nullptr;
    size_t len = 0;
    if (e2s_events_format(ev.data(), ev.size(), 1, &p, &text, &len)) {
        std::cerr << "ebwt2snp: " << e2s_last_error(nullptr) << std::endl;
        return 2;
    }
    const std::string out_path = input.substr(0, input.rfind(".fast")) + ".snp";
    const bool wrote = host::write_all(out_path, text, len);
    e2s_free(text);
    if (!wrote) {
        std::cerr << "ebwt2snp: cannot write " << out_path << std::endl;
        return 2;
    }
    return 0;
}

// -G > 1: one context per device used, every one with all the reads staged; the key cuts once, each shard's range built on its
// device, the halo rows collected here and applied, then ebwt2clust's multi-shard sequence (scan, e2s_exchange_finish, finalize)
// and clust2snp on every shard.  One thread per device: the builder sizes its work from the device's free memory, so two builds
// on one device must not overlap.  .clusters = every shard's head record, own records and tail records in shard order; the events
// in shard order, numbered across shards.
static int sharded(const std::string& input, const host::Reads& reads, int G, int x, int y, int z, uint32_t k, int min_len,
                   const e2s_snp_params& p) {
    const uint64_t n_reads = reads.n_reads();
    int n_dev = 0;
    if (e2s_device_count(&n_dev) || n_dev < 1) {
        std::cerr << "ebwt2snp: no CUDA device: " << e2s_last_error(nullptr) << std::endl;
        return 2;
    }
    const int D = n_dev < G ? n_dev : G;
    std::vector<e2s_ctx*> ctx(size_t(D), nullptr);
    std::vector<e2s_shard*> sh(size_t(G), nullptr);
    std::vector<int> rc(size_t(D), 0);
    std::vector<std::string> err(static_cast<size_t>(D));
    // fn(d) on every device at once, or fn(g) for every shard, the shards of one device one after another
    auto per_device = [&](const std::function<int(int)>& fn) {
        std::vector<std::thread> th;
        for (int d = 0; d < D; ++d)
            th.emplace_back([&, d]() {
                if (rc[size_t(d)]) return;
                rc[size_t(d)] = fn(d);
                if (rc[size_t(d)]) err[size_t(d)] = e2s_last_error(ctx[size_t(d)]);
            });
        for (auto& t : th) t.join();
        for (int d = 0; d < D; ++d)
            if (rc[size_t(d)]) {
                std::cerr << "ebwt2snp: GPU " << d << ": " << (err[size_t(d)].empty() ? e2s_last_error(nullptr) : err[size_t(d)].c_str()) << std::endl;
                return false;
            }
        return true;
    };
    auto per_shard = [&](const std::function<int(int)>& fn) {
        return per_device([&](int d) {
            int r = 0;
            for (int g = d; g < G && !r; g += D) r = fn(g);
            return r;
        });
    };
    if (!per_device([&](int d) {
            int r = e2s_ctx_create(d, &ctx[size_t(d)]);
            return r ? r : e2s_reads_stage(ctx[size_t(d)], reads.bases.data(), reads.off.data(), n_reads);
        }))
        return 2;
    std::vector<uint64_t> key_lo(static_cast<size_t>(G)), pos(static_cast<size_t>(G) + 1);
    if (e2s_reads_key_cuts(ctx[0], reads.off.data(), G, key_lo.data(), pos.data())) {
        std::cerr << "ebwt2snp: " << e2s_last_error(ctx[0]) << std::endl;
        return 2;
    }
    const uint64_t W = e2s_shard_halo_row_words();
    std::vector<uint64_t> rows(size_t(G) * W);
    if (!per_shard([&](int g) {
            e2s_ctx* c = ctx[size_t(g % D)];
            int r = e2s_shard_create(c, pos[size_t(g) + 1] - pos[size_t(g)], pos[size_t(g)], pos[size_t(G)], &sh[size_t(g)]);
            if (!r) r = e2s_shard_build_egsa_range(sh[size_t(g)], reads.off.data(), key_lo[size_t(g)], g + 1 < G ? key_lo[size_t(g) + 1] : 0, x, y, z);
            return r ? r : e2s_shard_halo_row(sh[size_t(g)], rows.data() + size_t(g) * W);
        }))
        return 2;
    host::stamp("key ranges built into the shards");
    std::vector<e2s_cluster_summary> sums(static_cast<size_t>(G));
    std::vector<e2s_stats> own(static_cast<size_t>(G));
    if (!per_shard([&](int g) {
            e2s_shard* s = sh[size_t(g)];
            int r = e2s_shard_halo_apply(s, rows.data(), G, g);
            if (!r) r = e2s_shard_seal(s);
            if (!r) r = e2s_cluster_prefilter(s, p.mcov_out);
            if (!r) r = e2s_cluster_run(s, k, min_len, &sums[size_t(g)]);
            return r ? r : e2s_statistics(s, &own[size_t(g)]);  // (before finalize: the shard's own records)
        }))
        return 2;
    std::vector<e2s_cluster_merged> mg(static_cast<size_t>(G));
    e2s_stats total;
    for (int g = 0; g < G; ++g)
        if (e2s_exchange_finish(sums.data(), own.data(), G, g, p.mcov_out, p.pval, &mg[size_t(g)], &total)) {
            std::cerr << "ebwt2snp: " << e2s_last_error(nullptr) << std::endl;
            return 2;
        }
    std::vector<std::vector<uint8_t>> rec10(static_cast<size_t>(G));
    std::vector<std::vector<e2s_event>> ev(static_cast<size_t>(G));
    std::vector<e2s_snp_counts> cnt(static_cast<size_t>(G));
    if (!per_shard([&](int g) {
            e2s_shard* s = sh[size_t(g)];
            uint64_t m = 0, nv = 0;
            int r = e2s_cluster_finalize(s, &mg[size_t(g)]);
            if (!r) r = e2s_find_events(s, &p, total.max_clust_length, &cnt[size_t(g)]);
            if (!r) r = e2s_cluster_count(s, &m);
            if (!r) {
                rec10[size_t(g)].resize(size_t(m) * 10 + 16);
                r = e2s_cluster_fetch_packed(s, rec10[size_t(g)].data(), m, &m);
                rec10[size_t(g)].resize(size_t(m) * 10);
            }
            if (!r) r = e2s_events_fetch(s, nullptr, 0, &nv);
            if (!r && nv) {
                ev[size_t(g)].resize(size_t(nv));
                r = e2s_events_fetch(s, ev[size_t(g)].data(), nv, &nv);
            }
            return r;
        }))
        return 2;
    host::stamp("clusters + events on the host");
    std::vector<uint8_t> all_rec;
    std::vector<e2s_event> all_ev;
    uint64_t n_candidates = 0;
    bool saw_n = false;
    for (int g = 0; g < G; ++g) {
        all_rec.insert(all_rec.end(), rec10[size_t(g)].begin(), rec10[size_t(g)].end());
        all_ev.insert(all_ev.end(), ev[size_t(g)].begin(), ev[size_t(g)].end());
        n_candidates += cnt[size_t(g)].n_candidates;
        saw_n = saw_n || cnt[size_t(g)].saw_n;
    }
    if (!host::write_all(input + ".clusters", all_rec.data(), all_rec.size())) {
        std::cerr << "ebwt2snp: cannot write " << input << ".clusters" << std::endl;
        return 2;
    }
    // the reference counts closures in an unsigned int (ref:ebwt2clust.cpp:88,137)
    std::cout << "Done. " << static_cast<unsigned int>(mg[size_t(G) - 1].n_clust_out) << " clusters saved to output file." << std::endl;
    const int wr = write_snp(input, all_ev, p, n_candidates, saw_n);
    if (wr) return wr;
    host::stamp(".clusters + .snp written");
    host::quick_exit_unless_asked(0);
    for (auto* s : sh) e2s_shard_destroy(s);
    for (auto* c : ctx) e2s_ctx_destroy(c);
    return 0;
}

int main(int argc, char** argv) {
    host::stamp("start");
    e2s_snp_params def;
    e2s_snp_default_params(&def);
    if (argc < 3) help();
    e2s_snp_params p;
    memset(&p, 0, sizeof p);
    int k = 0, min_len = 0, x = 0, y = 0, z = 0, max_snvs = 0, shards = 1;
    std::string input;
    int opt;
    while ((opt = getopt(argc, argv, "hi:n:p:v:L:R:m:g:c:x:y:z:e:k:l:G:")) != -1) {
        switch (opt) {
            case 'h': help(); break;
            case 'i': input = optarg; break;
            case 'n': p.nr_reads1 = uint64_t(int64_t(atoi(optarg))); break;
            case 'm': p.mcov_out = atoi(optarg); break;
            case 'g': p.max_gap = atoi(optarg); break;
            case 'L': p.k_left = atoi(optarg); break;
            case 'c': p.consensus_reads = atoi(optarg); break;
            case 'R': p.k_right = atoi(optarg); break;
            case 'p': p.pval = atof(optarg); break;
            case 'v': max_snvs = atoi(optarg); break;
            case 'e': p.max_err = int(atof(optarg)); break;
            case 'x': x = atoi(optarg); break;
            case 'y': y = atoi(optarg); break;
            case 'z': z = atoi(optarg); break;
            case 'k': k = atoi(optarg); break;
            case 'l': min_len = atoi(optarg); break;
            case 'G': shards = atoi(optarg); break;
            default: help();
        }
    }
    (void)max_snvs;  // parsed, never used, as by clust2snp (the test is against the default 3)
    // 0 means "use the default", for every option as in the two tools
    x = x == 0 ? 1 : x;
    y = y == 0 ? 4 : y;
    z = z == 0 ? 1 : z;
    k = k == 0 ? 16 : k;
    min_len = min_len == 0 ? 2 : min_len;
    p.max_err = p.max_err == 0 ? def.max_err : p.max_err;
    p.consensus_reads = p.consensus_reads == 0 ? def.consensus_reads : p.consensus_reads;
    p.max_gap = p.max_gap == 0 ? def.max_gap : p.max_gap;
    p.k_left = p.k_left == 0 ? def.k_left : p.k_left;
    p.k_right = p.k_right == 0 ? def.k_right : p.k_right;
    p.pval = p.pval == 0 ? def.pval : p.pval;
    p.mcov_out = p.mcov_out == 0 ? def.mcov_out : p.mcov_out;
    p.max_snvs = def.max_snvs;
    if (input.empty() || p.nr_reads1 == 0) help();
    auto ok = [](int v) { return v == 1 || v == 2 || v == 4 || v == 8; };
    if (!ok(x) || !ok(y) || !ok(z)) {
        std::cerr << "ebwt2snp: -x/-y/-z must be 1, 2, 4 or 8" << std::endl;
        return 2;
    }
    if (shards < 1) {
        std::cerr << "ebwt2snp: -G must be at least 1" << std::endl;
        return 2;
    }

    host::Reads reads;
    if (!reads.load(input) || reads.n_reads() == 0) {
        std::cout << "Error: could not read " << input << std::endl;
        return 1;
    }
    const uint64_t n_reads = reads.n_reads(), n = reads.bases.size() + n_reads;
    std::cout << "This is ebwt2snp. Input file: " << input << std::endl;
    host::stamp("FASTA parsed");

    if (shards > 1) return sharded(input, reads, shards, x, y, z, uint32_t(k), min_len, p);

    e2s_ctx* ctx = nullptr;
    e2s_shard* sh = nullptr;
    e2s_pipeline_result res;
    memset(&res, 0, sizeof res);
    int r = e2s_ctx_create(0, &ctx);
    if (!r) r = e2s_reads_stage(ctx, reads.bases.data(), reads.off.data(), n_reads);
    if (!r) r = e2s_shard_create(ctx, n, 0, n, &sh);
    if (!r) r = e2s_shard_build_egsa(sh, reads.off.data(), x, y, z);
    if (!r) r = e2s_shard_seal(sh);
    if (!r) host::stamp("index built into the shard + sealed");
    if (!r) r = e2s_pipeline_resident(sh, uint32_t(k), min_len, &p, &res);
    uint64_t m = 0, nv = 0;
    std::vector<uint8_t> rec10;
    std::vector<e2s_event> ev;
    if (!r) r = e2s_cluster_count(sh, &m);
    if (!r) {
        rec10.resize(size_t(m) * 10 + 16);
        r = e2s_cluster_fetch_packed(sh, rec10.data(), m, &m);
    }
    if (!r) r = e2s_events_fetch(sh, nullptr, 0, &nv);
    if (!r) {
        ev.resize(size_t(nv));
        if (nv) r = e2s_events_fetch(sh, ev.data(), nv, &nv);
    }
    if (r) {
        const char* e = ctx ? e2s_last_error(ctx) : "";
        std::cerr << "ebwt2snp: " << (e[0] ? e : e2s_last_error(nullptr)) << std::endl;
        return 2;
    }
    host::stamp("clusters + events on the host");

    if (!host::write_all(input + ".clusters", rec10.data(), size_t(m) * 10)) {
        std::cerr << "ebwt2snp: cannot write " << input << ".clusters" << std::endl;
        return 2;
    }
    // the reference counts closures in an unsigned int (ref:ebwt2clust.cpp:88,137)
    std::cout << "Done. " << static_cast<unsigned int>(res.n_clust_out) << " clusters saved to output file." << std::endl;
    ev.resize(size_t(nv));
    const int wr = write_snp(input, ev, p, res.snp.n_candidates, res.snp.saw_n != 0);
    if (wr) return wr;
    host::stamp(".clusters + .snp written");
    host::quick_exit_unless_asked(0);  // (everything is on disk: skip the teardown of the CUDA context unless E2S_CLI_CLEAN_EXIT is set)
    e2s_shard_destroy(sh);
    e2s_ctx_destroy(ctx);
    return 0;
}
