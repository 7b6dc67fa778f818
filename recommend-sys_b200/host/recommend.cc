// recommend.cc — top-N recommendation through the C++ mirror (core.hpp KNN::Recommend): fit one KNN estimator on
// a ratings file, then list the n best unrated items of each given user.
//
//   recommend <ratings file: user<TAB>item<TAB>rating per line> <cosine|msd|pearson> <basic|centered|zscore|baseline>
//             <userBased 0|1> <k> <n> <user> [<user> ...]
//   recommend ... <k> <n> --given <ratings file>   (KNN::RecommendGiven: the users of the second file, with the
//             ratings given there instead of the train set's; one line per user in order of first appearance)
//   recommend ... <k> <n> --update <ratings file> <user> [<user> ...]   (KNN::Update with the second file's ratings,
//             then KNN::Recommend)
//
// The estimator is fitted with k = 40 and `k` is set afterwards (Predict reads k at call time, core/knn.go:80-81).
// One output line per user: the user id, then n pairs "item score", the score as the 16 hex digits of its bits.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>

#include "core.hpp"

static core::DataSet load_file(const char *path) {  // core/data.go:287-310 (Atoi per field)
    core::DataSet d;
    std::ifstream f(path);
    if (!f) { std::fprintf(stderr, "cannot open %s\n", path); std::exit(1); }
    std::string line;
    while (std::getline(f, line)) {
        std::stringstream ss(line);
        std::string a, b, c;
        std::getline(ss, a, '\t'); std::getline(ss, b, '\t'); std::getline(ss, c, '\t');
        d.Users.push_back(std::atoll(a.c_str()));
        d.Items.push_back(std::atoll(b.c_str()));
        d.Ratings.push_back((double)std::atoll(c.c_str()));
    }
    return d;
}

int main(int argc, char **argv) {
    if (argc < 8) {
        std::fprintf(stderr, "usage: %s <ratings.tsv> <sim> <knn type> <userBased 0|1> <k> <n> <user>...\n", argv[0]);
        return 2;
    }
    const core::TrainSet train = core::NewTrainSet(load_file(argv[1]));
    core::Sim sim;
    if (!std::strcmp(argv[2], "cosine")) sim = core::Sim::Cosine;
    else if (!std::strcmp(argv[2], "msd")) sim = core::Sim::MSD;
    else if (!std::strcmp(argv[2], "pearson")) sim = core::Sim::Pearson;
    else { std::fprintf(stderr, "unknown sim %s\n", argv[2]); return 2; }
    core::KNN knn(argv[3], core::Parameters{{"sim", sim}, {"userBased", std::atoi(argv[4]) != 0}, {"k", 40}});
    knn.Fit(train);
    knn.Params.Set("k", std::atoi(argv[5]));
    const int n = std::atoi(argv[6]);
    std::vector<int64_t> users;
    std::vector<int64_t> items;
    std::vector<double> scores;
    if (!std::strcmp(argv[7], "--given") && argc == 9) {
        knn.RecommendGiven(load_file(argv[8]), n, users, items, scores);
    } else {
        int a = 7;
        if (!std::strcmp(argv[7], "--update") && argc >= 10) {
            knn.Update(load_file(argv[8]));
            a = 9;
        }
        for (; a < argc; a++) users.push_back(std::atoll(argv[a]));
        knn.Recommend(users, n, items, scores);
    }
    for (size_t u = 0; u < users.size(); u++) {
        std::printf("%" PRId64, users[u]);
        for (int x = 0; x < n; x++) {
            uint64_t bits;
            std::memcpy(&bits, &scores[u * n + x], 8);
            std::printf(" %" PRId64 " %016" PRIx64, items[u * n + x], bits);
        }
        std::printf("\n");
    }
    return 0;
}
