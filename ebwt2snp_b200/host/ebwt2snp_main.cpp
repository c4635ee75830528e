// ebwt2snp -- reads to SNPs in one process and one CUDA context: the FASTA's reads cross PCIe once, the index is built on the
// GPU straight into the resident shard that scans it (no X.gesa), then ebwt2clust and clust2snp run on that shard.  Writes the
// X.clusters and the .snp file that `build_gesa -x -y -z`, `ebwt2clust` and `clust2snp` with the same options write, and prints
// the counting lines of both tools.  The calls are those of e2s_pipeline_reads, made one by one so that the records and events
// are fetched at the sizes the step reports.  One GPU: the whole eBWT and the reads must fit it.
#include <getopt.h>

#include <iostream>

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
                 "\n"
                 "Builds the index on GPU 0 and keeps it there: no index file is written or read. One GPU only (E2S_GPUS is\n"
                 "ignored); the index takes 14.25 bytes per position on the device. For a larger index, several GPUs, reads\n"
                 "containing N or the BCR (-b) layout, run build_gesa, ebwt2clust and clust2snp.\n"
              << std::flush;
    exit(0);
}

int main(int argc, char** argv) {
    host::stamp("start");
    e2s_snp_params def;
    e2s_snp_default_params(&def);
    if (argc < 3) help();
    e2s_snp_params p;
    memset(&p, 0, sizeof p);
    int k = 0, min_len = 0, x = 0, y = 0, z = 0, max_snvs = 0;
    std::string input;
    int opt;
    while ((opt = getopt(argc, argv, "hi:n:p:v:L:R:m:g:c:x:y:z:e:k:l:")) != -1) {
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

    host::Reads reads;
    if (!reads.load(input) || reads.n_reads() == 0) {
        std::cout << "Error: could not read " << input << std::endl;
        return 1;
    }
    const uint64_t n_reads = reads.n_reads(), n = reads.bases.size() + n_reads;
    std::cout << "This is ebwt2snp. Input file: " << input << std::endl;
    host::stamp("FASTA parsed");

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
    std::cout << "Done. " << res.snp.n_candidates << " potential variants detected (some might be detected twice: on fw and rev strands)"
              << std::endl;
    if (res.snp.saw_n)
        std::cerr << "ebwt2snp: warning: N bases met; the reference maps them through rand() (ref:include.hpp:273), here they count as A" << std::endl;
    if (res.snp.n_candidates == 0) {  // clust2snp writes no .snp then either
        std::cerr << "ebwt2snp: no candidate variants; no .snp written" << std::endl;
        return 3;
    }
    char* text = nullptr;
    size_t len = 0;
    if (e2s_events_format(ev.data(), nv, 1, &p, &text, &len)) {
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
    host::stamp(".clusters + .snp written");
    host::quick_exit_unless_asked(0);  // (everything is on disk: skip the teardown of the CUDA context unless E2S_CLI_CLEAN_EXIT is set)
    e2s_shard_destroy(sh);
    e2s_ctx_destroy(ctx);
    return 0;
}
