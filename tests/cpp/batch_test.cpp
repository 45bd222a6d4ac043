// C++ user of the shim's batch calls: many (source, target) cloud pairs answered by knnBatch / matchBatch in one call
// each.  The pairs' descriptors come concatenated in two raw float32 dumps written by the pytest driver
// (tests/test_gpu_batch.py); results go back as text so the driver can compare every pair with the oracle.
//   batch_test <fpfh|shot|rops> <src.bin> <tgt.bin> <k> <out.txt> <n_src_0> <n_tgt_0> [<n_src_1> <n_tgt_1> ...]
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>

#include "b200match_shim.hpp"

using namespace b200match;

template <typename FeatureT>
static std::vector<FeatureT> load(std::ifstream &f, size_t n) {
    std::vector<FeatureT> v(n);
    f.read(reinterpret_cast<char *>(v.data()), (std::streamsize) (n * sizeof(FeatureT)));
    if (!f) throw std::runtime_error("descriptor dump is too short");
    return v;
}

template <typename FeatureT>
static int run(int argc, char **argv) {
    std::ifstream fs(argv[2], std::ios::binary), ft(argv[3], std::ios::binary);
    CloudPairs<FeatureT> pairs;
    for (int a = 6; a + 1 < argc; a += 2) {
        auto s = load<FeatureT>(fs, std::stoul(argv[a]));
        auto t = load<FeatureT>(ft, std::stoul(argv[a + 1]));
        pairs.emplace_back(std::move(s), std::move(t));
    }
    AlignmentParameters parameters;
    parameters.randomness = std::stoi(argv[4]);
    FILE *out = fopen(argv[5], "w");
    auto knn = knnBatch<FeatureT>(pairs, parameters);
    for (size_t p = 0; p < knn.size(); ++p) {
        if (knn[p].size() != pairs[p].first.size()) abort();
        for (size_t i = 0; i < knn[p].size(); ++i) {
            fprintf(out, "knn %zu %zu %zu", p, i, knn[p][i].match_indices.size());
            for (size_t m = 0; m < knn[p][i].match_indices.size(); ++m)
                fprintf(out, " %d %.9g", knn[p][i].match_indices[m], knn[p][i].distances[m]);
            fprintf(out, "\n");
        }
    }
    const struct { const char *name; int mode; } modes[] = {
        {"one_sided", B200M_MODE_ONE_SIDED}, {"mutual", B200M_MODE_MUTUAL}, {"ratio", B200M_MODE_RATIO}};
    for (const auto &m : modes) {
        BatchMatches r = matchBatch<FeatureT>(pairs, parameters, m.mode);
        for (size_t p = 0; p < r.correspondences.size(); ++p) {
            fprintf(out, "match %s %zu %zu %.9g\n", m.name, p, r.correspondences[p]->size(), r.average_distances[p]);
            for (const auto &c : *r.correspondences[p]) fprintf(out, "corr %s %zu %d %d %.9g\n", m.name, p, c.index_query, c.index_match, c.distance);
        }
    }
    fclose(out);
    return 0;
}

int main(int argc, char **argv) {
    if (argc < 8 || argc % 2 != 0) {
        std::cerr << "usage: batch_test <fpfh|shot|rops> src.bin tgt.bin k out.txt n_src_0 n_tgt_0 [n_src_1 n_tgt_1 ...]\n";
        return 2;
    }
    try {
        if (!strcmp(argv[1], "fpfh")) return run<FPFHSignature33>(argc, argv);
        if (!strcmp(argv[1], "shot")) return run<SHOT352>(argc, argv);
        if (!strcmp(argv[1], "rops")) return run<Histogram135>(argc, argv);
    } catch (const std::exception &e) {
        std::cerr << "error: " << e.what() << "\n";
        return 1;
    }
    return 2;
}
