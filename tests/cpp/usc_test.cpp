// C++ user of the shim with pcl::UniqueShapeContext1960 rows (7876 bytes: descriptor[1960], rf[9]): matchBF in both
// directions and the LeftToRightMatcher, as the reference's factory instantiates them for `descriptor_id: usc`.
// Descriptors come from a raw float32 dump written by the pytest driver (tests/test_gpu_long_descriptors.py), results
// go back as text so the driver can compare with the oracle.
//   usc_test <src.bin> <n_src> <tgt.bin> <n_tgt> <k> <out.txt>
#include <cstdio>
#include <fstream>
#include <iostream>

#include "b200match_shim.hpp"

using namespace b200match;
using FeatureT = UniqueShapeContext1960;

static std::vector<FeatureT> load(const char *path, size_t n) {
    std::vector<FeatureT> v(n);
    std::ifstream f(path, std::ios::binary);
    f.read(reinterpret_cast<char *>(v.data()), (std::streamsize) (n * sizeof(FeatureT)));
    if (!f) throw std::runtime_error(std::string("cannot read ") + path);
    return v;
}

int main(int argc, char **argv) {
    if (argc != 7) {
        std::cerr << "usage: usc_test <src.bin> <n_src> <tgt.bin> <n_tgt> <k> <out.txt>\n";
        return 2;
    }
    static_assert(FeatureT::descriptorSize() == 1960, "USC-1960 rows carry 1960 descriptor floats");
    if (feature_dim<FeatureT>() != 1960) abort();
    size_t ns = std::stoul(argv[2]), nt = std::stoul(argv[4]);
    auto src = load(argv[1], ns);
    auto tgt = load(argv[3], nt);
    AlignmentParameters parameters;
    parameters.randomness = std::stoi(argv[5]);
    FILE *out = fopen(argv[6], "w");
    for (int dir = 0; dir < 2; ++dir) {
        const auto &q = dir ? tgt : src;
        const auto &t = dir ? src : tgt;
        auto bf = matchBF<FeatureT>(q, t, parameters);
        if (bf.size() != q.size()) abort();
        for (size_t i = 0; i < q.size(); ++i) {
            fprintf(out, "knn %d %zu %zu", dir, i, bf[i].match_indices.size());
            for (size_t m = 0; m < bf[i].match_indices.size(); ++m)
                fprintf(out, " %d %.9g", bf[i].match_indices[m], bf[i].distances[m]);
            fprintf(out, "\n");
        }
    }
    // the LeftToRightMatcher on one scale, keypoints on the lattice the driver builds too
    auto lattice = [](size_t n, float step) {
        std::vector<float> xyz(4 * n, 0.f);
        for (size_t i = 0; i < n; ++i) {
            xyz[4 * i + 0] = step * (float) (i % 17);
            xyz[4 * i + 1] = step * (float) ((i / 17) % 13);
            xyz[4 * i + 2] = step * (float) (i / 221);
        }
        return xyz;
    };
    const auto sx = lattice(ns, 0.5f), tx = lattice(nt, 0.25f);
    using Impl = FeatureBasedMatcherImpl<FeatureT>;
    parameters.matching_id = "lr";
    auto matcher = getFeatureBasedMatcherFromParameters<FeatureT>(Impl::makeStorage(src, sx.data(), 16, 0.3f),
                                                                  Impl::makeStorage(tgt, tx.data(), 16, 0.2f), parameters);
    auto corrs = matcher->match();
    fprintf(out, "matcher lr %s %zu %.9g\n", matcher->getClassName().c_str(), corrs->size(), matcher->getAverageDistance());
    for (const auto &c : *corrs) fprintf(out, "corr lr %d %d %.9g\n", c.index_query, c.index_match, c.distance);
    fclose(out);
    return 0;
}
