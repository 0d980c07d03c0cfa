// komb2 — drop-in replacement for the reference's komb2 executable
// (reference src/komb2.cpp): same flags, same stage order, same stdout stage
// lines, same three output files (edgelist.txt, kcore.tsv, CoreA_anomaly.txt);
// the graph build, k-core and CORE-A run on a B200 through libkombgpu's C ABI.
// KOMB.py (reference KOMB.py:435-462) drives it unchanged.
//
// Environment: KOMB_GPU_DEVICE (CUDA ordinal, default 0);
//              KOMB_GPU_DEVICES=0,1,... (two or more ordinals: the graph is partitioned over these GPUs of the node,
//              one host thread per GPU, peer-memory path of libkombgpu; same output files);
//              KOMB_COREA_KEY=exact64 selects the overflow-free CORE-A key
//              (default "ref32" reproduces the reference's int32 wrap, quirk Q5);
//              KOMB_TOKENIZE=host tokenises and interns the SAM text on the host (default: on the device,
//              kombgpu_sam_parse with one GPU, kombgpu_dist_sam_parse over the ranks with KOMB_GPU_DEVICES);
//              KOMB_OUTPUT=host formats the three files on the host (default with device tokenisation: on the device,
//              kombgpu_graph_format with one GPU, each rank's slice with kombgpu_dist_graph_format with KOMB_GPU_DEVICES;
//              with KOMB_TOKENIZE=host always on the host); KOMB_TIMING=1 prints wall-clock marks;
//              KOMB_UNITIG_FASTA=anomalous, =truss or =anomalous,truss also writes the -u FASTA's records of the
//              anomalous unitigs (CORE-A above the IQR fence q3 + 1.5 (q3 - q1)) to <outdir>/anomalous_unitigs.fasta and
//              of the unitigs on the max-truss edges of the maximal core to <outdir>/truss_unitigs.fasta, indexed, joined
//              and copied on the device (truss needs one GPU: not with KOMB_GPU_DEVICES).  Unset, the FASTA is only
//              opened, as the reference does.
//              KOMB_ONION=1 also writes <outdir>/onion.tsv after kcore.tsv: every unitig's onion layer (the layers of a
//              synchronous k-core peel, kombgpu_graph_onion) as "#VID\tName\tCoreness\tLayer" rows, formatted where the
//              other files are (one GPU only: not with KOMB_GPU_DEVICES).
#include <omp.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "cli.hpp"
#include "kgraph.hpp"

#define KOMB2_VERSION "2.0"

int main(int argc, const char **argv) {
    omp_set_dynamic(0);
    auto begin = std::chrono::steady_clock::now();
    const komb::Options opt = komb::parse_cli(argc, argv, KOMB2_VERSION, omp_get_max_threads());

    const char *dev_env = getenv("KOMB_GPU_DEVICE");
    const char *key_env = getenv("KOMB_COREA_KEY");
    const int device = dev_env ? atoi(dev_env) : 0;
    const int key_mode = (key_env && strcmp(key_env, "exact64") == 0) ? KOMBGPU_KEY_EXACT64 : KOMBGPU_KEY_REF32;

    std::vector<int> devices;
    if (const char *list = getenv("KOMB_GPU_DEVICES")) {
        for (const char *p = list; *p;) {
            char *end = nullptr;
            const long d = strtol(p, &end, 10);
            if (end == p) break;
            devices.push_back((int)d);
            p = *end == ',' ? end + 1 : end;
        }
    }

    // checked before any device work
    bool fasta_anomalous = false, fasta_truss = false;
    if (const char *uf = getenv("KOMB_UNITIG_FASTA")) {
        const std::string list(uf);
        for (size_t b = 0; b <= list.size();) {
            size_t e = list.find(',', b);
            if (e == std::string::npos) e = list.size();
            const std::string w = list.substr(b, e - b);
            if (w == "anomalous") fasta_anomalous = true;
            else if (w == "truss") fasta_truss = true;
            else if (!(w.empty() && list.empty())) {
                fprintf(stderr, "komb2: KOMB_UNITIG_FASTA=%s: unknown word '%s' (expected anomalous, truss or anomalous,truss)\n", uf, w.c_str());
                return EXIT_FAILURE;
            }
            b = e + 1;
        }
        if (fasta_truss && devices.size() > 1) {
            fprintf(stderr, "komb2: KOMB_UNITIG_FASTA=%s: truss_unitigs.fasta needs one GPU (the graph partitioned over KOMB_GPU_DEVICES has "
                            "no truss)\n", uf);
            return EXIT_FAILURE;
        }
    }

    bool onion = false;
    if (const char *on = getenv("KOMB_ONION")) {
        if (strcmp(on, "1") == 0) onion = true;
        else if (on[0] && strcmp(on, "0") != 0) {
            fprintf(stderr, "komb2: KOMB_ONION=%s: expected 1 (write onion.tsv) or 0\n", on);
            return EXIT_FAILURE;
        }
        if (onion && devices.size() > 1) {
            fprintf(stderr, "komb2: KOMB_ONION=1: onion.tsv needs one GPU (the graph partitioned over KOMB_GPU_DEVICES has no onion "
                            "layers)\n");
            return EXIT_FAILURE;
        }
    }

    komb::Kgraph kg((uint32_t)opt.threads, (uint64_t)opt.readlen, device, key_mode, devices);
    kg.setUnitigFasta(fasta_anomalous, fasta_truss, opt.input_unitigs);
    kg.setOnion(onion);
    komb::HitTable hits;
    komb::MappedFile sam1, sam2;  // the hit table points into these until the ids exist
    auto begin_komb = std::chrono::steady_clock::now();

    kg.readSAM(opt.input, sam1, hits, opt.fulgor);
    kg.readSAM(opt.input2, sam2, hits, opt.fulgor);
    auto post_sam = std::chrono::steady_clock::now();
    fprintf(stdout, "\nTime elapsed for reading SAMs: %.3f s\n",
            std::chrono::duration_cast<std::chrono::microseconds>(post_sam - begin_komb).count() / 1000000.0);

    kg.getEdgeInfo(hits);
    auto post_edgeinfo = std::chrono::steady_clock::now();
    fprintf(stdout, "\nTime elapsed for edgeInfo: %.3f s\n",
            std::chrono::duration_cast<std::chrono::microseconds>(post_edgeinfo - post_sam).count() / 1000000.0);

    kg.generateGraph(hits);
    auto post_generate = std::chrono::steady_clock::now();
    fprintf(stdout, "\nTime elapsed for generateGraph: %.3f s\n",
            std::chrono::duration_cast<std::chrono::microseconds>(post_generate - post_edgeinfo).count() / 1000000.0);

    kg.readEdgeList(opt.output, opt.input_unitigs, hits);
    fprintf(stdout, "Created Kcore\n");
    auto post_core = std::chrono::steady_clock::now();
    // the reference labels this stage "edgeInfo" as well (src/komb2.cpp:124)
    fprintf(stdout, "\nTime elapsed for edgeInfo: %.3f s\n",
            std::chrono::duration_cast<std::chrono::microseconds>(post_core - post_generate).count() / 1000000.0);
    fprintf(stdout, "\nTime elapsed for combineFile: %.3f s\n", 0.0);

    kg.anomalyDetection(opt.output, true, opt.input_unitigs, hits);
    fprintf(stdout, "\nTime elapsed for anomalyDetection: %.3f s\n", komb::seconds_since(post_core));
    fprintf(stdout, "Identified anomalous unitigs\n");
    fprintf(stdout, "Created anomalouss unitigs file\n");
    fprintf(stdout, "\nTime elapsed for KOMB: %.3f s\n", komb::seconds_since(begin_komb));
    fprintf(stdout, "\nTime elapsed for analysis (sec) = %.3f \n", komb::seconds_since(begin));
    return 0;
}
