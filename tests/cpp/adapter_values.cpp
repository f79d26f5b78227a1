// Runs include/sfe_adapter.hpp on cases that Python writes as raw little-endian arrays, and writes the raw results back, so
// that tests/test_call_surfaces.py can compare them value by value with the oracle.  The mocks expose the reference's accessor
// names as in adapter_test.cpp, except that Frame::GetIndex reports the map points of an in-frame set (src/matcher.cpp:144)
// and every Mappoint sits at an array slot chosen by Python: std::set<Mappoint*> then iterates in slot order.
// The test compiles it into a temporary directory (g++ -std=c++14 -pthread adapter_values.cpp libsfe.so).
//
// usage: adapter_values proj    <dir>            meta.txt xw.f64 mpdesc.u8 inframe.u8 slot.i32 kps.kp kdesc.u8 -> out.i32
//        adapter_values extract <dir>            meta.txt l.u8 r.u8                                          -> out.bin
//        adapter_values threads <projdir> <extractdir> <iters>   both cases on two threads, compared with one pass
//
// proj meta.txt:    n m width height fx fy cx cy d0 d1 d2 d3 calls, then per call: qx qy qz qw tx ty tz radius
//   out.i32 = calls x m: the Python index of the map point matched to each keypoint, or -1
// extract meta.txt: width height step nfeatures scale_factor nlevels ini_th_fast min_th_fast
//   out.bin = four blocks [int32 n][n x 28 B keypoints][n x 32 B descriptors]: extract(L), extract(R) and the left and right
//   results of extractStereo(L, R); then [int32 n][n x int32] stereo indices of extractStereo
#define SFE_ADAPTER_CV_STANDIN
#include "cv_standin.hpp"
#include "../../include/sfe_adapter.hpp"

#include <cstdio>
#include <fstream>
#include <iterator>
#include <thread>

struct Vec3 { double v[3]; double operator[](int i) const { return v[i]; } };
struct Quat { double x_, y_, z_, w_; double x() const { return x_; } double y() const { return y_; } double z() const { return z_; } double w() const { return w_; } };
struct SE3 { Quat r; Vec3 t; const Quat &rotation() const { return r; } const Vec3 &translation() const { return t; } };  // g2o::SE3Quat's accessors
struct KMat { double k[3][3]; double operator()(int r, int c) const { return k[r][c]; } };
struct DVec { double d[4]; double operator()(int i) const { return d[i]; } };
struct Camera {
    KMat K; DVec D; int w, h;
    const KMat &GetK() const { return K; } const DVec &GetD() const { return D; }
    int GetWidth() const { return w; } int GetHeight() const { return h; }
};
struct Mappoint {
    int id = -1;  // index on the Python side
    Vec3 X{};
    cv::Mat desc;
    Vec3 GetXw() const { return X; } cv::Mat GetDescription() const { return desc; }
};
struct Frame {
    std::vector<cv::KeyPoint> keypoints_;
    cv::Mat descriptions_;
    std::set<const Mappoint *> in_frame;
    Camera cam;
    const std::vector<cv::KeyPoint> &GetKeypoints() const { return keypoints_; }
    const cv::Mat GetDescription(int i) const { return descriptions_.row(i); }
    int GetIndex(const Mappoint *mp) const { return in_frame.count(mp) ? 0 : -1; }
    const Camera *GetCamera() const { return &cam; }
};

static std::vector<uint8_t> slurp(const std::string &path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error("cannot read " + path);
    return std::vector<uint8_t>(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
}

static void dump(const std::string &path, const void *p, size_t n) {
    std::ofstream f(path, std::ios::binary);
    f.write((const char *)p, (std::streamsize)n);
    if (!f) throw std::runtime_error("cannot write " + path);
}

struct ProjCase {
    std::vector<Mappoint> slots;  // slots[slot[i]] = map point i
    std::vector<uint8_t> mp_desc, kdesc;
    Frame frame;
    std::vector<std::pair<SE3, double>> calls;

    explicit ProjCase(const std::string &dir) {
        std::ifstream meta(dir + "/meta.txt");
        int n = 0, m = 0, calls_n = 0;
        Camera &c = frame.cam;
        double fx, fy, cx, cy;
        meta >> n >> m >> c.w >> c.h >> fx >> fy >> cx >> cy >> c.D.d[0] >> c.D.d[1] >> c.D.d[2] >> c.D.d[3] >> calls_n;
        if (!meta) throw std::runtime_error("bad proj meta.txt");
        c.K = KMat{{{fx, 0, cx}, {0, fy, cy}, {0, 0, 1}}};
        for (int i = 0; i < calls_n; i++) {
            SE3 T;
            double r;
            meta >> T.r.x_ >> T.r.y_ >> T.r.z_ >> T.r.w_ >> T.t.v[0] >> T.t.v[1] >> T.t.v[2] >> r;
            calls.push_back({T, r});
        }
        if (!meta) throw std::runtime_error("bad proj meta.txt");
        const std::vector<uint8_t> xw = slurp(dir + "/xw.f64"), in = slurp(dir + "/inframe.u8"), sl = slurp(dir + "/slot.i32"),
                                   kps = slurp(dir + "/kps.kp");
        mp_desc = slurp(dir + "/mpdesc.u8");
        kdesc = slurp(dir + "/kdesc.u8");
        if (xw.size() != (size_t)n * 24 || mp_desc.size() != (size_t)n * 32 || in.size() != (size_t)n || sl.size() != (size_t)n * 4 ||
            kps.size() != (size_t)m * 28 || kdesc.size() != (size_t)m * 32)
            throw std::runtime_error("proj case: array sizes do not match meta.txt");
        slots.resize(n);
        for (int i = 0; i < n; i++) {
            int32_t s;
            std::memcpy(&s, &sl[(size_t)i * 4], 4);
            if (s < 0 || s >= n || slots[s].id >= 0) throw std::runtime_error("slot.i32 is not a permutation");
            Mappoint &p = slots[s];
            p.id = i;
            std::memcpy(p.X.v, &xw[(size_t)i * 24], 24);
            p.desc = cv::Mat(1, 32, CV_8U, &mp_desc[(size_t)i * 32]);
            if (in[i]) frame.in_frame.insert(&p);
        }
        frame.keypoints_.resize(m);
        if (m) std::memcpy((void *)frame.keypoints_.data(), kps.data(), kps.size());
        frame.descriptions_ = cv::Mat(m, 32, CV_8U, kdesc.data());
    }

    // one int32 per (call, keypoint)
    std::vector<int32_t> run() const {
        std::set<Mappoint *> mps;
        for (const Mappoint &p : slots) mps.insert(const_cast<Mappoint *>(&p));
        const size_t m = frame.keypoints_.size();
        std::vector<int32_t> out(calls.size() * m, -1);
        for (size_t c = 0; c < calls.size(); c++) {
            const std::map<int, Mappoint *> got = sfe_adapter::ProjectionMatch(mps, calls[c].first, &frame, calls[c].second);
            for (const auto &kv : got) {
                if (kv.first < 0 || (size_t)kv.first >= m) throw std::runtime_error("ProjectionMatch returned a keypoint out of range");
                out[c * m + (size_t)kv.first] = kv.second->id;
            }
        }
        return out;
    }
};

struct ExtractCase {
    int w = 0, h = 0, step = 0, nfeatures = 0, nlevels = 0, ini = 0, mn = 0;
    float scale = 0;
    std::vector<uint8_t> L, R;  // step-strided rows; the padding bytes are filled with garbage that must not be read

    explicit ExtractCase(const std::string &dir) {
        std::ifstream meta(dir + "/meta.txt");
        meta >> w >> h >> step >> nfeatures >> scale >> nlevels >> ini >> mn;
        if (!meta || step < w) throw std::runtime_error("bad extract meta.txt");
        const std::vector<uint8_t> l = slurp(dir + "/l.u8"), r = slurp(dir + "/r.u8");
        if (l.size() != (size_t)w * h || r.size() != l.size()) throw std::runtime_error("extract case: image sizes do not match meta.txt");
        L.assign((size_t)step * h, 0xA5);
        R.assign((size_t)step * h, 0x5A);
        for (int y = 0; y < h; y++) {
            std::memcpy(&L[(size_t)y * step], &l[(size_t)y * w], w);
            std::memcpy(&R[(size_t)y * step], &r[(size_t)y * w], w);
        }
    }

    static void put(std::vector<uint8_t> &o, const void *p, size_t n) { o.insert(o.end(), (const uint8_t *)p, (const uint8_t *)p + n); }
    static void put_features(std::vector<uint8_t> &o, const std::vector<cv::KeyPoint> &k, const cv::Mat &d) {
        const int32_t n = (int32_t)k.size();
        if (d.rows != (d.empty() ? 0 : n)) throw std::runtime_error("descriptor rows differ from the keypoint count");
        put(o, &n, 4);
        put(o, k.data(), k.size() * sizeof(cv::KeyPoint));
        for (int i = 0; i < n; i++) put(o, d.ptr(i), 32);
    }

    std::vector<uint8_t> run(ORB_SLAM2::ORBextractor &ex) const {
        cv::Mat l(h, w, CV_8UC1, (void *)L.data(), (size_t)step), r(h, w, CV_8UC1, (void *)R.data(), (size_t)step);
        std::vector<cv::KeyPoint> k[4];
        cv::Mat d[4];
        std::vector<int> sidx;
        ex.extract(l, cv::noArray(), k[0], d[0]);
        ex.extract(r, cv::noArray(), k[1], d[1]);
        ex.extractStereo(l, r, k[2], d[2], k[3], d[3], sidx);
        std::vector<uint8_t> o;
        for (int i = 0; i < 4; i++) put_features(o, k[i], d[i]);
        const int32_t ns = (int32_t)sidx.size();
        put(o, &ns, 4);
        put(o, sidx.data(), sidx.size() * 4);
        return o;
    }
    std::unique_ptr<ORB_SLAM2::ORBextractor> make() const {
        return std::unique_ptr<ORB_SLAM2::ORBextractor>(new ORB_SLAM2::ORBextractor(nfeatures, scale, nlevels, ini, mn));
    }
};

int main(int argc, char **argv) {
    if (argc < 3) return 2;
    const std::string mode = argv[1];
    try {
        if (mode == "proj") {
            const ProjCase pc(argv[2]);
            const std::vector<int32_t> out = pc.run();
            dump(std::string(argv[2]) + "/out.i32", out.data(), out.size() * 4);
            printf("calls=%zu keypoints=%zu\n", pc.calls.size(), pc.frame.keypoints_.size());
        } else if (mode == "extract") {
            const ExtractCase ec(argv[2]);
            const std::vector<uint8_t> out = ec.run(*ec.make());
            dump(std::string(argv[2]) + "/out.bin", out.data(), out.size());
            printf("bytes=%zu\n", out.size());
        } else if (mode == "threads") {
            // "one handle per thread" (include/sfe.h, sfe_adapter::thread_matcher): two threads, each with its own matcher and
            // extractor, repeat both cases; every result must equal the single-threaded pass
            if (argc < 5) return 2;
            const ProjCase pc(argv[2]);
            const ExtractCase ec(argv[3]);
            const int iters = atoi(argv[4]);
            const std::vector<int32_t> want_p = pc.run();
            const std::vector<uint8_t> want_e = ec.run(*ec.make());
            dump(std::string(argv[2]) + "/out.i32", want_p.data(), want_p.size() * 4);
            dump(std::string(argv[3]) + "/out.bin", want_e.data(), want_e.size());
            int diff[2] = {0, 0};
            std::string err[2];
            auto worker = [&](int t) {
                try {
                    std::unique_ptr<ORB_SLAM2::ORBextractor> ex = ec.make();
                    for (int i = 0; i < iters; i++) {
                        diff[t] += pc.run() != want_p;
                        diff[t] += ec.run(*ex) != want_e;
                    }
                } catch (const std::exception &e) {
                    err[t] = e.what();
                }
            };
            std::thread a(worker, 0), b(worker, 1);
            a.join();
            b.join();
            for (int t = 0; t < 2; t++)
                if (!err[t].empty()) throw std::runtime_error("thread " + std::to_string(t) + ": " + err[t]);
            printf("iters=%d diff0=%d diff1=%d\n", iters, diff[0], diff[1]);
        } else {
            return 2;
        }
    } catch (const std::exception &e) {
        printf("exception: %s\n", e.what());
        return 1;
    }
    return 0;
}
