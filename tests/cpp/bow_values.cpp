// Runs the BoW path of include/sfe_adapter.hpp -- Vocabulary::loadFromTextFile, transform, and Database::add / query -- on
// inputs that Python writes, and writes the raw results back, so that tests/test_bow_database.py can compare them with the
// oracle.  The test compiles it into a temporary directory (g++ -std=c++14 -pthread bow_values.cpp libsfe.so).
//
// usage: bow_values query  <dir>   voc.txt (DBoW2 text format) desc.bin queries.txt -> bow.txt results.txt
//        bow_values reject <voc>   constructs a Database on a vocabulary whose header names another scoring type
//
// desc.bin:    int32 images, then per image int32 n and n x 32 descriptor bytes
// queries.txt: lines "max_results max_id"; every image's BowVector is queried with each line after all images were added
// bow.txt:     per image "n id bits id bits ..." (bits = the value's IEEE double as 16 hex digits)
// results.txt: per (image, line of queries.txt) "image max_results max_id n entry bits entry bits ..."
#define SFE_ADAPTER_CV_STANDIN
#include "cv_standin.hpp"
#include "../../include/sfe_adapter.hpp"

#include <cinttypes>
#include <cstdio>
#include <fstream>

// DBoW2::Result / QueryResults stand-ins: what queryL1 constructs (Result(EntryId, double)) and pushes back
struct Result {
    unsigned int Id;
    double Score;
    Result(unsigned int id, double score) : Id(id), Score(score) {}
};
struct QueryResults : public std::vector<Result> {};
typedef std::map<unsigned int, double> BowVector;                   // DBoW2::BowVector
typedef std::map<unsigned int, std::vector<unsigned int>> FeatureVector;  // DBoW2::FeatureVector

static uint64_t bits(double x) {
    uint64_t u;
    std::memcpy(&u, &x, 8);
    return u;
}

static int run_query(const std::string &dir) {
    sfe_adapter::Vocabulary voc;
    if (!voc.loadFromTextFile(dir + "/voc.txt")) {
        std::fprintf(stderr, "cannot load %s/voc.txt\n", dir.c_str());
        return 1;
    }
    std::ifstream f(dir + "/desc.bin", std::ios::binary);
    int32_t images = 0;
    f.read((char *)&images, 4);
    std::vector<BowVector> bows(images);
    sfe_adapter::Database db(voc);
    FILE *bo = std::fopen((dir + "/bow.txt").c_str(), "w");
    for (int i = 0; i < images; i++) {
        int32_t n = 0;
        f.read((char *)&n, 4);
        std::vector<uint8_t> raw((size_t)n * 32);
        f.read((char *)raw.data(), (std::streamsize)raw.size());
        std::vector<cv::Mat> feats;
        for (int j = 0; j < n; j++) feats.push_back(cv::Mat(1, 32, 0, raw.data() + (size_t)j * 32));
        FeatureVector fv;
        voc.transform(feats, bows[i], fv, 4);
        std::fprintf(bo, "%zu", bows[i].size());
        for (const auto &kv : bows[i]) std::fprintf(bo, " %u %016" PRIx64, kv.first, bits(kv.second));
        std::fprintf(bo, "\n");
        const unsigned int id = db.add(bows[i]);
        if (id != (unsigned int)i || db.size() != (unsigned int)i + 1) {
            std::fprintf(stderr, "add returned %u (size %u) for image %d\n", id, db.size(), i);
            return 1;
        }
    }
    std::fclose(bo);
    std::ifstream qf(dir + "/queries.txt");
    std::vector<std::pair<int, int>> qs;
    int k = 0, max_id = 0;
    while (qf >> k >> max_id) qs.emplace_back(k, max_id);
    FILE *ro = std::fopen((dir + "/results.txt").c_str(), "w");
    for (int i = 0; i < images; i++) {
        for (const auto &p : qs) {
            QueryResults ret;
            ret.push_back(Result(12345, 1.0));  // query() starts from an empty list, as DBoW2's does
            db.query(bows[i], ret, p.first, p.second);
            std::fprintf(ro, "%d %d %d %zu", i, p.first, p.second, ret.size());
            for (const Result &r : ret) std::fprintf(ro, " %u %016" PRIx64, r.Id, bits(r.Score));
            std::fprintf(ro, "\n");
        }
    }
    std::fclose(ro);
    return 0;
}

static int run_reject(const std::string &path) {
    sfe_adapter::Vocabulary voc;
    if (!voc.loadFromTextFile(path)) {
        std::fprintf(stderr, "cannot load %s\n", path.c_str());
        return 1;
    }
    try {
        sfe_adapter::Database db(voc);
    } catch (const std::runtime_error &e) {
        std::printf("rejected=%s\n", e.what());
        return 0;
    }
    std::printf("accepted\n");
    return 0;
}

int main(int argc, char **argv) {
    if (argc != 3) {
        std::fprintf(stderr, "usage: bow_values query <dir> | reject <voc.txt>\n");
        return 2;
    }
    const std::string mode = argv[1];
    try {
        if (mode == "query") return run_query(argv[2]);
        if (mode == "reject") return run_reject(argv[2]);
    } catch (const std::exception &e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 2;
}
