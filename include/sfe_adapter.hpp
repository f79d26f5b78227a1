// sfe_adapter.hpp -- header-only C++ host side above the sfe C ABI that keeps the reference's own
// call surface, so frame.cpp / posetracker.cpp / pipeline.cpp / loopcloser.cpp compile unchanged:
//
//   ORB_SLAM2::ORBextractor          replaces include/orb_extractor.h:45-133 + src/orb_extractor.cpp
//   sfe_adapter::StereoMatch         body for  void StereoMatch(StereoFrame*)          (src/matcher.cpp:54-132)
//   sfe_adapter::ProjectionMatch     body for  std::map<int,Mappoint*> ProjectionMatch (src/matcher.cpp:134-209)
//
// It is written against the OpenCV 3.4 types the reference uses (cv::Mat, cv::KeyPoint,
// cv::InputArray, cv::OutputArray).  Where OpenCV is not installed (this repo's CI) define
// SFE_ADAPTER_CV_STANDIN before including it and provide the few members used below
// (tests/cpp/cv_standin.hpp does).  The matcher templates only touch the reference's public
// accessors (GetKeypoints, GetDescription(i), GetCamera()->GetK(), mp->GetXw(), ...), so they bind to
// the real Frame / StereoFrame / Mappoint / g2o::SE3Quat as they are.
//
// Errors: an empty image returns silently with the outputs untouched (src/orb_extractor.cpp:1046-1047);
// zero keypoints releases the descriptor matrix (:1064-1065); every other failure throws
// std::runtime_error carrying sfe_last_error().  There is no CPU fallback.
#ifndef SFE_ADAPTER_HPP_
#define SFE_ADAPTER_HPP_

#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "sfe.h"

#ifndef SFE_ADAPTER_CV_STANDIN
#include <opencv2/core/core.hpp>
#include <opencv2/features2d/features2d.hpp>
#endif

static_assert(sizeof(sfe_keypoint) == 28, "sfe_keypoint must be 28 bytes");
static_assert(sizeof(cv::KeyPoint) == sizeof(sfe_keypoint), "cv::KeyPoint layout changed: adapter memcpy is invalid");

namespace sfe_adapter {

inline void check(int status, const char *what) {
    if (status != SFE_OK)
        throw std::runtime_error(std::string(what) + ": " + sfe_status_string(status) + " (" + sfe_last_error() + ")");
}

// one matcher handle per thread: ProjectionMatch is entered from the tracking AND the mapping
// thread of the reference (src/pipeline.cpp:98-141, src/posetracker.cpp:186), handles are not re-entrant
inline sfe_matcher *thread_matcher(int device = 0) {
    struct Holder {
        sfe_matcher *m = nullptr;
        ~Holder() { sfe_matcher_destroy(m); }
    };
    static thread_local Holder h;
    if (!h.m) check(sfe_matcher_create(device, &h.m), "sfe_matcher_create");
    return h.m;
}

}  // namespace sfe_adapter

namespace sfe_adapter {
// Staging array in pinned host memory (sfe_host_alloc): a one-image / one-pair call then has its results stored straight into
// it by one kernel instead of several DMA copies.  Grows, never shrinks; contents are not preserved.
template <typename T>
class PinnedArray {
public:
    PinnedArray() = default;
    ~PinnedArray() { if (p_) sfe_host_free(p_); }
    PinnedArray(const PinnedArray &) = delete;
    PinnedArray &operator=(const PinnedArray &) = delete;
    void resize(size_t n) {
        if (n <= cap_) return;
        if (p_) sfe_host_free(p_);
        p_ = nullptr; cap_ = 0;
        void *q = nullptr;
        check(sfe_host_alloc(&q, n * sizeof(T)), "sfe_host_alloc");
        p_ = static_cast<T *>(q); cap_ = n;
    }
    T *data() { return p_; }
    const T *data() const { return p_; }
private:
    T *p_ = nullptr;
    size_t cap_ = 0;
};
}  // namespace sfe_adapter

namespace ORB_SLAM2 {

class ORBextractor {
public:
    enum { HARRIS_SCORE = 0, FAST_SCORE = 1 };

    ORBextractor(int nfeatures, float scaleFactor, int nlevels, int iniThFAST, int minThFAST)
        : nfeatures_(nfeatures), scaleFactor_(scaleFactor), nlevels_(nlevels) {
        sfe_extractor_params p = {nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST};
        sfe_adapter::check(sfe_extractor_create(&p, 0, 2, &ex_), "sfe_extractor_create");
        sfe_adapter::check(sfe_extractor_max_keypoints(ex_, &cap_), "sfe_extractor_max_keypoints");
        mvScaleFactor.resize(nlevels); mvInvScaleFactor.resize(nlevels);
        mvLevelSigma2.resize(nlevels); mvInvLevelSigma2.resize(nlevels);
        sfe_adapter::check(sfe_extractor_tables(ex_, mvScaleFactor.data(), mvInvScaleFactor.data(), mvLevelSigma2.data(),
                                                mvInvLevelSigma2.data(), nullptr), "sfe_extractor_tables");
        kps_.resize(cap_);
    }
    ~ORBextractor() { sfe_extractor_destroy(ex_); }
    ORBextractor(const ORBextractor &) = delete;
    ORBextractor &operator=(const ORBextractor &) = delete;

    // Compute the ORB features and descriptors on an image.  Mask is ignored (as in the reference).
    void extract(cv::InputArray _image, cv::InputArray /*mask*/, std::vector<cv::KeyPoint> &_keypoints,
                 cv::OutputArray _descriptors) {
        if (_image.empty()) return;
        cv::Mat image = _image.getMat();
        if (image.type() != CV_8UC1) throw std::invalid_argument("ORBextractor::extract: CV_8UC1 image expected");
        int need = 0;  // a very wide image can return more than the default bound (4 * nIni nodes per level)
        sfe_adapter::check(sfe_extractor_max_keypoints_for(ex_, image.cols, image.rows, &need), "sfe_extractor_max_keypoints_for");
        if (need > cap_) { cap_ = need; kps_.resize(cap_); }
        desc_.resize((size_t)cap_ * 32);
        counts_.resize(2);
        int32_t &n = counts_.data()[0];
        n = 0;
        sfe_adapter::check(sfe_extract_batch(ex_, image.data, (size_t)image.step * image.rows, 1, image.cols, image.rows, (int)image.step,
                                             kps_.data(), desc_.data(), cap_, &n), "sfe_extract");
        if (n == 0) {
            _descriptors.release();
        } else {
            _descriptors.create(n, 32, CV_8U);
            cv::Mat d = _descriptors.getMat();
            for (int i = 0; i < n; i++) std::memcpy(d.ptr(i), desc_.data() + (size_t)i * 32, 32);
        }
        _keypoints.resize(n);
        if (n) std::memcpy((void *)_keypoints.data(), kps_.data(), sizeof(sfe_keypoint) * (size_t)n);
    }

    int inline GetLevels() { return nlevels_; }
    float inline GetScaleFactor() { return (float)scaleFactor_; }
    std::vector<float> inline GetScaleFactors() { return mvScaleFactor; }
    std::vector<float> inline GetInverseScaleFactors() { return mvInvScaleFactor; }
    std::vector<float> inline GetScaleSigmaSquares() { return mvLevelSigma2; }
    std::vector<float> inline GetInverseScaleSigmaSquares() const { return mvInvLevelSigma2; }

    // The reference exposes the pyramid as a public member that nothing outside the extractor reads
    // (grep mvImagePyramid: orb_extractor.* only).  It stays declared for source compatibility and is
    // left empty: the pyramid lives in HBM.
    std::vector<cv::Mat> mvImagePyramid;

    static int DescriptorDistance(const cv::Mat &a, const cv::Mat &b) { return sfe_hamming256(a.data, b.data); }

    sfe_extractor *handle() { return ex_; }

    // The keyframe path of StereoFrame in ONE call -- extract(left) (src/frame.cpp:47), extract(right) (:388) and
    // StereoMatch (src/pipeline.cpp:248) -- with a single upload / download round trip instead of three; same results.
    // stereo_indices is what StereoMatch hands to SetStereoCorrespond.  (An addition to the reference's surface for
    // callers that hold both images; the three separate calls keep working.)
    void extractStereo(cv::InputArray _left, cv::InputArray _right, std::vector<cv::KeyPoint> &kps_l, cv::OutputArray _desc_l,
                       std::vector<cv::KeyPoint> &kps_r, cv::OutputArray _desc_r, std::vector<int> &stereo_indices) {
        if (_left.empty() || _right.empty()) return;
        cv::Mat L = _left.getMat(), R = _right.getMat();
        if (L.type() != CV_8UC1 || R.type() != CV_8UC1 || L.rows != R.rows || L.cols != R.cols || L.step != R.step)
            throw std::invalid_argument("ORBextractor::extractStereo: two CV_8UC1 images of the same geometry expected");
        int need = 0;
        sfe_adapter::check(sfe_extractor_max_keypoints_for(ex_, L.cols, L.rows, &need), "sfe_extractor_max_keypoints_for");
        if (need > cap_) { cap_ = need; kps_.resize(cap_); }
        desc_.resize((size_t)cap_ * 32);
        kps_r_.resize(cap_); desc_r_.resize((size_t)cap_ * 32); sidx_.resize(cap_);
        counts_.resize(2);
        int32_t *nl = counts_.data(), *nr = counts_.data() + 1;
        sfe_adapter::check(sfe_stereo_frames(ex_, L.data, R.data, (size_t)L.step * L.rows, 1, L.cols, L.rows, (int)L.step, nullptr,
                                             kps_.data(), desc_.data(), nl, kps_r_.data(), desc_r_.data(), nr, sidx_.data(), nullptr,
                                             cap_), "sfe_stereo_frames");
        fill(kps_, desc_, *nl, kps_l, _desc_l);
        fill(kps_r_, desc_r_, *nr, kps_r, _desc_r);
        stereo_indices.assign(sidx_.data(), sidx_.data() + *nl);
    }

protected:
    int nfeatures_;
    double scaleFactor_;
    int nlevels_;
    std::vector<float> mvScaleFactor, mvInvScaleFactor, mvLevelSigma2, mvInvLevelSigma2;

private:
    static void fill(const sfe_adapter::PinnedArray<sfe_keypoint> &k, const sfe_adapter::PinnedArray<uint8_t> &d, int n,
                     std::vector<cv::KeyPoint> &kps, cv::OutputArray desc) {
        if (n == 0) {
            desc.release();
        } else {
            desc.create(n, 32, CV_8U);
            cv::Mat m = desc.getMat();
            for (int i = 0; i < n; i++) std::memcpy(m.ptr(i), d.data() + (size_t)i * 32, 32);
        }
        kps.resize(n);
        if (n) std::memcpy((void *)kps.data(), k.data(), sizeof(sfe_keypoint) * (size_t)n);
    }
    sfe_extractor *ex_ = nullptr;
    int cap_ = 0;
    sfe_adapter::PinnedArray<sfe_keypoint> kps_, kps_r_;
    sfe_adapter::PinnedArray<uint8_t> desc_, desc_r_;
    sfe_adapter::PinnedArray<int32_t> sidx_, counts_;
};

}  // namespace ORB_SLAM2

namespace sfe_adapter {

// void StereoMatch(StereoFrame* frame)  -- include/matcher.h:33
template <class StereoFrameT>
void StereoMatch(StereoFrameT *frame) {
    const std::vector<cv::KeyPoint> &kl = frame->GetKeypoints();
    const std::vector<cv::KeyPoint> &kr = frame->GetRightKeypoints();
    std::vector<uint8_t> dl(kl.size() * 32), dr(kr.size() * 32);
    for (size_t i = 0; i < kl.size(); i++) std::memcpy(&dl[i * 32], frame->GetDescription((int)i).data, 32);
    for (size_t j = 0; j < kr.size(); j++) std::memcpy(&dr[j * 32], frame->GetRightDescription((int)j).data, 32);
    std::vector<int> stereo_indices(kl.size(), -1);
    const sfe_stereo_params sp = {3., 100., 0.5};  // src/matcher.cpp:68-70
    static_assert(sizeof(int) == sizeof(int32_t), "int must be 32 bit");
    check(sfe_stereo_match(thread_matcher(), (const sfe_keypoint *)kl.data(), dl.data(), (int)kl.size(),
                           (const sfe_keypoint *)kr.data(), dr.data(), (int)kr.size(), &sp, stereo_indices.data(), nullptr),
          "sfe_stereo_match");
    frame->SetStereoCorrespond(stereo_indices);
}

// std::map<int, Mappoint*> ProjectionMatch(const std::set<Mappoint*>&, const g2o::SE3Quat&, const Frame*, double)
//   -- include/matcher.h:35-38.  PoseT needs rotation() -> a quaternion with x(), y(), z(), w() and translation()
//   (g2o::SE3Quat has both); the pose travels as that unit quaternion + translation and the device evaluates
//   predicted_Tcw * Xw the way g2o / Eigen do (sfe_se3), so boundary points fall on the reference's side.
template <class MappointT, class PoseT, class FrameT>
std::map<int, MappointT *> ProjectionMatch(const std::set<MappointT *> &mappoints, const PoseT &predicted_Tcw,
                                           const FrameT *curr_frame, double search_radius) {
    const double best12_threshold = 0.5;  // src/matcher.cpp:138
    const auto *camera = curr_frame->GetCamera();
    std::vector<MappointT *> order;  // the set's iteration order = the reference's query order (T3)
    std::vector<double> xw;
    std::vector<uint8_t> desc, skip;
    order.reserve(mappoints.size());
    for (MappointT *mp : mappoints) {
        order.push_back(mp);
        const auto X = mp->GetXw();
        xw.push_back(X[0]); xw.push_back(X[1]); xw.push_back(X[2]);
        const cv::Mat d = mp->GetDescription();
        desc.insert(desc.end(), d.data, d.data + 32);
        skip.push_back(curr_frame->GetIndex(mp) >= 0 ? 1 : 0);  // :144
    }
    const auto &q = predicted_Tcw.rotation();
    const auto &t = predicted_Tcw.translation();
    const sfe_se3 Tcw = {q.x(), q.y(), q.z(), q.w(), t[0], t[1], t[2]};
    sfe_camera cam;
    const auto &K = camera->GetK();
    const auto &D = camera->GetD();
    cam.fx = K(0, 0); cam.fy = K(1, 1); cam.cx = K(0, 2); cam.cy = K(1, 2);
    for (int i = 0; i < 4; i++) cam.d[i] = D(i);
    cam.width = camera->GetWidth();
    cam.height = camera->GetHeight();
    const std::vector<cv::KeyPoint> &kps = curr_frame->GetKeypoints();
    std::vector<uint8_t> kdesc(kps.size() * 32);
    for (size_t i = 0; i < kps.size(); i++) std::memcpy(&kdesc[i * 32], curr_frame->GetDescription((int)i).data, 32);
    std::vector<int32_t> to_query(kps.size(), -1);
    check(sfe_projection_match_se3(thread_matcher(), xw.data(), desc.data(), skip.data(), (int)order.size(), &Tcw, &cam,
                                   (const sfe_keypoint *)kps.data(), kdesc.data(), (int)kps.size(), search_radius,
                                   best12_threshold, to_query.data(), nullptr),
          "sfe_projection_match_se3");
    std::map<int, MappointT *> matches;
    for (size_t j = 0; j < kps.size(); j++)
        if (to_query[j] >= 0) matches[(int)j] = order[(size_t)to_query[j]];
    return matches;
}

// ORB_SLAM2::ORBVocabulary stand-in for Frame::ComputeBoW (src/frame.cpp:419-427): loads the DBoW2 text format
// (TemplatedVocabulary::loadFromTextFile, thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1338-1421), keeps the tree on the
// device and fills DBoW2::BowVector / DBoW2::FeatureVector (any std::map<unsigned, double> /
// std::map<unsigned, std::vector<unsigned>>) with transform()'s exact results: the descent runs on the GPU, the maps are
// built on the host in the reference's order of operations (sfe_bow_assemble).
class Vocabulary {
public:
    Vocabulary() = default;
    ~Vocabulary() { sfe_vocab_destroy(voc_); }
    Vocabulary(const Vocabulary &) = delete;
    Vocabulary &operator=(const Vocabulary &) = delete;

    bool loadFromTextFile(const std::string &filename) {
        std::ifstream f(filename.c_str());
        if (!f.good()) return false;
        std::string line;
        std::getline(f, line);
        int n1 = -1, n2 = -1;
        {
            std::stringstream ss(line);
            ss >> k_ >> L_ >> n1 >> n2;
        }
        if (k_ < 0 || k_ > 20 || L_ < 1 || L_ > 10 || n1 < 0 || n1 > 5 || n2 < 0 || n2 > 3) return false;
        std::vector<int32_t> parent(1, 0);
        std::vector<uint8_t> is_leaf(1, 0), desc(32, 0);
        std::vector<double> weight(1, 0.);
        while (std::getline(f, line)) {
            if (line.empty()) continue;
            std::stringstream ss(line);
            int pid = 0, leaf = 0;
            ss >> pid >> leaf;
            parent.push_back(pid);
            is_leaf.push_back(leaf > 0);
            for (int i = 0; i < 32; i++) {
                int v = 0;
                ss >> v;
                desc.push_back((uint8_t)v);
            }
            double w = 0.;
            ss >> w;
            weight.push_back(w);
        }
        return create(parent, is_leaf, desc, weight, L_, n1, n2);
    }

    // the arrays loadFromTextFile would have read; scoring / weighting = DBoW2::ScoringType / WeightingType values
    bool create(const std::vector<int32_t> &parent, const std::vector<uint8_t> &is_leaf, const std::vector<uint8_t> &desc,
                const std::vector<double> &weight, int L, int scoring, int weighting) {
        sfe_vocab_destroy(voc_);
        voc_ = nullptr;
        L_ = L;
        scoring_ = scoring;
        weighting_ = weighting;
        norm_ = scoring == 5 ? 0 : (scoring == 1 ? 2 : 1);  // ScoringObject.h:74-89: DOT_PRODUCT none, L2_NORM L2, the rest L1
        return sfe_vocab_create(thread_matcher(), (int)parent.size(), parent.data(), is_leaf.data(), desc.data(), weight.data(), L,
                                &voc_) == SFE_OK;
    }

    bool empty() const { return voc_ == nullptr; }
    int getScoringType() const { return scoring_; }
    // number of words (TemplatedVocabulary::size)
    unsigned int size() const {
        int n = 0;
        if (voc_) check(sfe_vocab_words(voc_, &n), "sfe_vocab_words");
        return (unsigned int)n;
    }

    // void transform(const std::vector<TDescriptor>& features, BowVector &v, FeatureVector &fv, int levelsup) const
    template <class BowVectorT, class FeatureVectorT>
    void transform(const std::vector<cv::Mat> &features, BowVectorT &v, FeatureVectorT &fv, int levelsup) const {
        v.clear();
        fv.clear();
        if (empty() || features.empty()) return;
        const int n = (int)features.size();
        std::vector<uint8_t> desc((size_t)n * 32);
        for (int i = 0; i < n; i++) std::memcpy(&desc[(size_t)i * 32], features[i].data, 32);
        std::vector<int32_t> wid(n), nid(n), ids(n);
        std::vector<double> w(n), vals(n);
        check(sfe_vocab_transform(thread_matcher(), voc_, desc.data(), n, levelsup, wid.data(), w.data(), nid.data()),
              "sfe_vocab_transform");
        int m = 0;
        check(sfe_bow_assemble(wid.data(), w.data(), n, weighting_, norm_, ids.data(), vals.data(), n, &m), "sfe_bow_assemble");
        for (int i = 0; i < m; i++) v[(unsigned)ids[i]] = vals[i];
        for (int i = 0; i < n; i++)
            if (w[i] > 0) fv[(unsigned)nid[i]].push_back((unsigned)i);
    }

private:
    sfe_vocab *voc_ = nullptr;
    int k_ = 0, L_ = 0, scoring_ = 0, weighting_ = 0, norm_ = 1;
};

// DBoW2::TemplatedDatabase stand-in for the loop-candidate query (thirdparty/DBoW2/DBoW2/TemplatedDatabase.h: add, query
// with L1 scoring = queryL1, size): the keyframe BowVectors stay on the device and every query is scored there, bit for bit.
// Equal scores come back in ascending entry id.  BowVectorT = any std::map<unsigned, double> (DBoW2::BowVector);
// QueryResultsT = a vector of a type constructible from (EntryId, double score) (DBoW2::QueryResults of DBoW2::Result).
// Only L1 scoring exists (ORBvoc.txt is "10 6 0 0"): a vocabulary with another scoring type is rejected.  One Database may
// be used from several threads (each call uses its thread's matcher handle).  There is no direct index (FeatureVector).
class Database {
public:
    typedef unsigned int EntryId;

    explicit Database(const Vocabulary &voc) {
        if (voc.empty()) throw std::invalid_argument("sfe_adapter::Database: empty vocabulary");
        if (voc.getScoringType() != 0)
            throw std::runtime_error(std::string("sfe_adapter::Database: ") + sfe_status_string(SFE_ERR_UNSUPPORTED) +
                                     " (only L1_NORM scoring is implemented)");
        check(sfe_bowdb_create(thread_matcher(), (int)voc.size(), &db_), "sfe_bowdb_create");
    }
    ~Database() { sfe_bowdb_destroy(db_); }
    Database(const Database &) = delete;
    Database &operator=(const Database &) = delete;

    template <class BowVectorT>
    EntryId add(const BowVectorT &v) {
        std::vector<int32_t> ids;
        std::vector<double> vals;
        flatten(v, ids, vals);
        const int64_t off[2] = {0, (int64_t)ids.size()};
        int32_t first = 0;
        check(sfe_bowdb_add(thread_matcher(), db_, off, ids.data(), vals.data(), 1, &first), "sfe_bowdb_add");
        return (EntryId)first;
    }

    // void query(const BowVector &vec, QueryResults &ret, int max_results = 1, int max_id = -1) const
    // 1 <= max_results <= SFE_BOWDB_MAX_RESULTS (DBoW2's "max_results <= 0: every entry" is not offered).
    template <class BowVectorT, class QueryResultsT>
    void query(const BowVectorT &vec, QueryResultsT &ret, int max_results = 1, int max_id = -1) const {
        ret.clear();
        std::vector<int32_t> ids;
        std::vector<double> vals;
        flatten(vec, ids, vals);
        const int64_t off[2] = {0, (int64_t)ids.size()};
        const int k = max_results;
        std::vector<int32_t> ent(k > 0 ? k : 1);
        std::vector<double> sc(k > 0 ? k : 1);
        int32_t n = 0;
        check(sfe_bowdb_query(thread_matcher(), db_, off, ids.data(), vals.data(), 1, max_id, k, ent.data(), sc.data(), &n, nullptr, 0),
              "sfe_bowdb_query");
        ret.reserve(n);
        for (int i = 0; i < n; i++) ret.push_back(typename QueryResultsT::value_type((EntryId)ent[i], sc[i]));
    }

    unsigned int size() const {
        int n = 0;
        check(sfe_bowdb_size(db_, &n), "sfe_bowdb_size");
        return (unsigned int)n;
    }

private:
    template <class BowVectorT>
    static void flatten(const BowVectorT &v, std::vector<int32_t> &ids, std::vector<double> &vals) {
        ids.reserve(v.size());
        vals.reserve(v.size());
        for (const auto &kv : v) {
            ids.push_back((int32_t)kv.first);
            vals.push_back((double)kv.second);
        }
    }
    sfe_bowdb *db_ = nullptr;
};

}  // namespace sfe_adapter

#endif  // SFE_ADAPTER_HPP_
