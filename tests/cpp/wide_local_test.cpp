// C++ user of the shim's guessed matchers: reference-shaped matchers with AlignmentParameters::guess set (one guess per
// cloud pair), answered by matchMany in one call and by each matcher's match().  The pairs come in one binary dump written
// by the pytest driver (tests/test_gpu_wide_local.py); per pair:
//   int32 n_scales, n_src_kps, n_tgt_kps; float iss_radius_src, iss_radius_tgt; float guess[16] (row-major)
//   per scale: int32 n_src, n_tgt; float32 src rows [n_src][33]; int32 src map [n_src]; float32 tgt rows; int32 tgt map
//   float32 src keypoints [n_src_kps][4]; float32 tgt keypoints [n_tgt_kps][4]
// Results go back as text; the moved keypoints the shim used (source by the guess, target by its inverse, [n][4] each,
// pair by pair) go to <out.txt>.moved, so the oracle can be fed the same coordinates.
//   wide_local_test <one_sided|lr|cluster> <k> <pairs.bin> <n_pairs> <radius> <out.txt>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>

#include "b200match_shim.hpp"

using namespace b200match;
using Matcher = FeatureBasedMatcherImpl<FPFHSignature33>;

template <typename T>
static std::vector<T> load(std::ifstream &f, size_t n) {
    std::vector<T> v(n);
    f.read(reinterpret_cast<char *>(v.data()), (std::streamsize) (n * sizeof(T)));
    if (!f) throw std::runtime_error("pair dump is too short");
    return v;
}

int main(int argc, char **argv) {
    if (argc != 7) {
        std::cerr << "usage: wide_local_test <one_sided|lr|cluster> <k> <pairs.bin> <n_pairs> <radius> <out.txt>\n";
        return 2;
    }
    try {
        AlignmentParameters params;
        params.matching_id = argv[1];
        params.randomness = atoi(argv[2]);
        params.cluster_k = 40;
        params.match_search_radius = (float) atof(argv[5]);
        std::ifstream in(argv[3], std::ios::binary);
        const int n_pairs = atoi(argv[4]);
        std::vector<std::vector<float>> xyz(2 * n_pairs);   // the Storages point into these
        std::vector<std::shared_ptr<Matcher>> ms;
        FILE *mv = fopen((std::string(argv[6]) + ".moved").c_str(), "wb");
        for (int p = 0; p < n_pairs; ++p) {
            const auto hdr = load<int32_t>(in, 3);
            const auto radii = load<float>(in, 2);
            const auto g = load<float>(in, 16);
            std::array<float, 16> guess;
            std::copy(g.begin(), g.end(), guess.begin());
            Matcher::Storage st[2];
            for (int s = 0; s < hdr[0]; ++s) {
                const auto n = load<int32_t>(in, 2);
                for (int side = 0; side < 2; ++side) {
                    st[side].kps_features_multiscale.push_back(load<FPFHSignature33>(in, (size_t) n[side]));
                    const auto map = load<int32_t>(in, (size_t) n[side]);
                    st[side].kps_indices_multiscale.emplace_back(map.begin(), map.end());
                }
            }
            for (int side = 0; side < 2; ++side) {
                xyz[2 * p + side] = load<float>(in, (size_t) hdr[1 + side] * 4);
                st[side].kps_xyz = xyz[2 * p + side].data();
                st[side].n_kps = (size_t) hdr[1 + side];
                st[side].kps_stride_bytes = 16;
                st[side].min_log2_radius = 0;
                st[side].max_log2_radius = hdr[0] - 1;
                st[side].iss_radius = radii[side];
                std::vector<float> moved(xyz[2 * p + side].size(), 0.f);
                moveKeypoints(st[side].kps_xyz, st[side].n_kps, 4, side ? invertGuess(guess) : guess, moved.data(), 4);
                fwrite(moved.data(), sizeof(float), moved.size(), mv);
            }
            AlignmentParameters pp = params;
            pp.guess = guess;
            FeatureBasedMatcher::Ptr m = getFeatureBasedMatcherFromParameters<FPFHSignature33>(st[0], st[1], pp);
            ms.push_back(std::dynamic_pointer_cast<Matcher>(m));
        }
        fclose(mv);
        const std::vector<CorrespondencesPtr> got = matchMany<FPFHSignature33>(ms);
        std::vector<float> avg;
        for (auto &m : ms) avg.push_back(m->getAverageDistance());
        FILE *o = fopen(argv[6], "w");
        for (int p = 0; p < n_pairs; ++p) {
            const CorrespondencesPtr one = ms[p]->match();   // the per-pair call
            bool same = one->size() == got[p]->size() && ms[p]->getAverageDistance() == avg[p];
            for (size_t i = 0; same && i < one->size(); ++i)
                same = memcmp(&(*one)[i], &(*got[p])[i], sizeof(Correspondence)) == 0;
            fprintf(o, "pair %d %zu %.9g %d\n", p, got[p]->size(), avg[p], same ? 1 : 0);
            for (const Correspondence &c : *got[p])
                fprintf(o, "corr %d %d %d %.9g %.9g\n", p, c.index_query, c.index_match, c.distance, c.threshold);
        }
        fclose(o);
        try {   // guessed and unguessed matchers are refused together
            std::vector<std::shared_ptr<Matcher>> mixed{ms[0], std::dynamic_pointer_cast<Matcher>(
                                                                   getFeatureBasedMatcherFromParameters<FPFHSignature33>(
                                                                       Matcher::makeStorage({}), Matcher::makeStorage({}), params))};
            matchMany<FPFHSignature33>(mixed);
            std::cerr << "a mix of guessed and unguessed matchers was accepted\n";
            return 1;
        } catch (const std::runtime_error &e) {
            if (std::string(e.what()).find("a guess or none") == std::string::npos) throw;
        }
    } catch (const std::exception &e) {
        std::cerr << e.what() << "\n";
        return 1;
    }
    return 0;
}
