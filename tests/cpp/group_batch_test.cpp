// matchMany on several GPUs: the same OneSided / LeftToRight / ClusterMatchers, guessed and not, answered with
// AlignmentParameters::devices = {0, .., n-1} (the pairs spread over the GPUs, b200m_group_match_multiscale[_local]_batch)
// and with devices = {0} (one context) must give byte-identical correspondences and averages.
//   group_batch_test <n_gpus>          exit 0: every comparison equal
#include <cstdio>
#include <cstring>
#include <iostream>
#include <random>

#include "b200match_shim.hpp"

using namespace b200match;
using Matcher = FeatureBasedMatcherImpl<FPFHSignature33>;

struct Cloud {
    std::vector<FPFHSignature33> desc;
    std::vector<float> xyz;   // [n][4]
};

static Cloud make_cloud(std::mt19937 &rng, size_t n) {
    std::uniform_real_distribution<float> u(0.f, 1.f);
    Cloud c;
    c.desc.resize(n);
    c.xyz.resize(n * 4, 0.f);
    for (size_t i = 0; i < n; ++i) {
        for (float &h : c.desc[i].histogram) h = 100.f * u(rng) * u(rng);
        for (int d = 0; d < 3; ++d) c.xyz[i * 4 + d] = 4.f * u(rng);
    }
    return c;
}

static std::vector<std::shared_ptr<Matcher>> make_matchers(const std::vector<Cloud> &clouds, const std::string &id, bool guessed,
                                                           const std::vector<int> &devices) {
    std::vector<std::shared_ptr<Matcher>> ms;
    for (size_t p = 0; p + 1 < clouds.size(); p += 2) {
        AlignmentParameters a;
        a.matching_id = id;
        a.randomness = 2;
        a.cluster_k = 40;
        a.devices = devices;
        if (guessed) {
            const float t = 0.05f * (float) p;
            a.guess = std::array<float, 16>{1.f, 0.f, 0.f, t, 0.f, 1.f, 0.f, -t, 0.f, 0.f, 1.f, 0.5f * t, 0.f, 0.f, 0.f, 1.f};
            a.match_search_radius = 1.5f;
        }
        auto src = Matcher::makeStorage(clouds[p].desc, clouds[p].xyz.data(), 16, 0.05f);
        auto tgt = Matcher::makeStorage(clouds[p + 1].desc, clouds[p + 1].xyz.data(), 16, 0.06f);
        ms.push_back(std::dynamic_pointer_cast<Matcher>(getFeatureBasedMatcherFromParameters<FPFHSignature33>(src, tgt, a)));
    }
    return ms;
}

int main(int argc, char **argv) {
    if (argc != 2) {
        std::cerr << "usage: group_batch_test <n_gpus>\n";
        return 2;
    }
    const int n_gpus = atoi(argv[1]);
    try {
        std::mt19937 rng(7);
        std::vector<Cloud> clouds;
        for (int i = 0; i < 14; ++i) clouds.push_back(make_cloud(rng, i == 2 ? 2500 : 300 + 40 * (size_t) i));
        std::vector<int> all;
        for (int d = 0; d < n_gpus; ++d) all.push_back(d);
        int bad = 0;
        for (const char *id : {"one_sided", "lr", "cluster"})
            for (bool guessed : {false, true}) {
                auto one = make_matchers(clouds, id, guessed, {0});
                auto many = make_matchers(clouds, id, guessed, all);
                const auto a = matchMany<FPFHSignature33>(one), b = matchMany<FPFHSignature33>(many);
                size_t n = 0;
                for (size_t p = 0; p < a.size(); ++p) {
                    bool same = a[p]->size() == b[p]->size() && one[p]->getAverageDistance() == many[p]->getAverageDistance();
                    for (size_t i = 0; same && i < a[p]->size(); ++i) same = memcmp(&(*a[p])[i], &(*b[p])[i], sizeof(Correspondence)) == 0;
                    if (!same) {
                        std::cerr << id << (guessed ? " guessed" : "") << ": pair " << p << " differs\n";
                        ++bad;
                    }
                    n += a[p]->size();
                }
                printf("%s%s: %zu pairs, %zu correspondences, devices {0} == %d devices\n", id, guessed ? " guessed" : "", a.size(), n, n_gpus);
                if (!n) ++bad;
            }
        return bad ? 1 : 0;
    } catch (const std::exception &e) {
        std::cerr << e.what() << "\n";
        return 1;
    }
}
