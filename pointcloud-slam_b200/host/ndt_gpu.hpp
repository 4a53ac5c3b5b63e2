// b200reg host adaptor — pclomp::NormalDistributionsTransform's interface on top of the C ABI.
//
// Mirrors pointcloud_match/ndt_omp/include/pclomp/ndt_omp.h:117-261 and the pcl::Registration calls the reference
// makes on it (jueying_slam/src/mapOptmization.cpp:683-693, localization.cpp:162-188,317-340): setInputTarget,
// setInputSource, align, hasConverged, getFinalTransformation, getTransformationProbability, getFinalNumIteration,
// setResolution / setStepSize / setOutlierRatio / setTransformationEpsilon / setMaximumIterations /
// setNeighborhoodSearchMethod / setNumThreads, calculateScore.  CloudT is any type with a `.points` vector of
// structs starting with float x, y, z (pcl::PointCloud<pcl::PointXYZI> qualifies) - PCL itself is not needed.
// 4x4 transforms are float[16] column-major, i.e. Eigen::Matrix4f::data().
#pragma once
#include <memory>
#include <stdexcept>
#include <vector>

#include "ivox_gpu.hpp"

namespace b200host {

enum NeighborSearchMethod { KDTREE, DIRECT26, DIRECT7, DIRECT1 };  // ndt_omp.h:61-66

template <typename CloudT>
class NormalDistributionsTransform {
   public:
    explicit NormalDistributionsTransform(int device = 0) : device_(device) {
        // constructor defaults, ndt_omp_impl.hpp:47-65
        prm_.resolution = 1.0f; prm_.step_size = 0.1; prm_.outlier_ratio = 0.55; prm_.trans_eps = 0.1;
        prm_.max_iter = 35; prm_.search = 7; prm_.min_pts = 6; prm_.eig_ratio = 0.01;
        for (int i = 0; i < 16; ++i) final_[i] = (i % 5 == 0) ? 1.f : 0.f;
    }
    ~NormalDistributionsTransform() { b200_ndt_destroy(ndt_); }

    void setResolution(float r) { prm_.resolution = r; dirty_ = true; }               // ndt_omp.h:142
    void setStepSize(double s) { prm_.step_size = s; dirty_ = true; }                  // :166
    void setOutlierRatio(double o) { prm_.outlier_ratio = o; dirty_ = true; }          // :184
    void setTransformationEpsilon(double e) { prm_.trans_eps = e; dirty_ = true; }     // pcl::Registration
    void setMaximumIterations(int n) { prm_.max_iter = n; dirty_ = true; }             // pcl::Registration
    void setNumThreads(int) {}                                                         // :117, the device decides
    void setNeighborhoodSearchMethod(NeighborSearchMethod m) {                         // :189
        prm_.search = m == KDTREE ? 0 : m == DIRECT1 ? 1 : m == DIRECT26 ? 27 : 7;
        dirty_ = true;
    }
    void setInputTarget(const std::shared_ptr<const CloudT>& cloud) { target_ = cloud; target_dirty_ = true; }   // :125-130
    void setInputSource(const std::shared_ptr<const CloudT>& cloud) { source_ = cloud; source_dirty_ = true; }

    /// align(output, guess): output = source transformed by the final transformation (pcl::Registration::align)
    void align(CloudT& output, const float* guess16 = nullptr) {
        sync();
        float I[16];
        for (int i = 0; i < 16; ++i) I[i] = (i % 5 == 0) ? 1.f : 0.f;
        int32_t rc = b200_ndt_align(ndt_, guess16 ? guess16 : I, final_, &result_);
        check(rc, "b200_ndt_align");
        output = *source_;
        for (auto& p : output.points) {
            const float x = p.x, y = p.y, z = p.z;
            p.x = final_[0] * x + final_[4] * y + final_[8] * z + final_[12];
            p.y = final_[1] * x + final_[5] * y + final_[9] * z + final_[13];
            p.z = final_[2] * x + final_[6] * y + final_[10] * z + final_[14];
        }
    }
    bool hasConverged() const { return result_.converged != 0; }
    const float* getFinalTransformation() const { return final_; }                        // column-major 4x4
    double getTransformationProbability() const { return result_.trans_probability; }   // ndt_omp.h:200-204
    int getFinalNumIteration() const { return result_.iters; }                            // :226-230
    double getMaxEigen() const {                                                          // :209-223 (localization-lost heuristic)
        double v = 0;
        check(b200_ndt_max_eigen(result_.hessian, &v), "b200_ndt_max_eigen");
        return v;
    }
    const double* getHessian() const { return result_.hessian; }
    /// pcl::Registration::getFitnessScore(max_range): mean squared nearest-neighbour distance after the last align
    double getFitnessScore(double max_range = 1.7976931348623157e308) {
        double s = 0;
        int64_t nr = 0;
        check(b200_ndt_fitness_score(ndt_, final_, max_range, &s, &nr), "b200_ndt_fitness_score");
        return s;
    }

    /// calculateScore (ndt_omp_impl.hpp:836-880) for h candidate poses (h x 16 floats, column-major)
    void calculateScore(const float* poses16, int64_t h, double* scores) {
        sync();
        check(b200_ndt_score_batch(ndt_, poses16, h, scores), "b200_ndt_score_batch");
    }
    /// Global relocalization with refinement (b200_reloc_refine): the top_k hypotheses of highest calculateScore (poses16 =
    /// this rank's slice, h x 16 column-major; local i = global h_begin + i * h_stride) are aligned from their poses and the
    /// converged one with the highest transformation probability wins.  comm may be NULL; with one, every rank passes the
    /// same top_k and max_range.  Returns the winning hypothesis (-1: none had a finite score) and fills the candidates in
    /// order (score descending, index ascending); `converged` = false when no candidate converged.  Errors throw.
    int64_t relocalizeRefine(b200_comm* comm, const float* poses16, int64_t h, int64_t h_begin, int64_t h_stride, int64_t top_k,
                             std::vector<b200_reloc_candidate>& candidates, bool* converged = nullptr,
                             double max_range = 1.7976931348623157e308) {
        sync();
        candidates.assign(top_k > 0 ? (size_t)top_k : 0, b200_reloc_candidate{});
        int64_t best = -1, n = 0;
        const int32_t rc = b200_reloc_refine(comm, ndt_, poses16, h, h_begin, h_stride, top_k, max_range, &best,
                                             candidates.empty() ? nullptr : candidates.data(), &n, nullptr);
        check(rc, "b200_reloc_refine");
        candidates.resize((size_t)n);
        if (converged) *converged = rc == B200_OK;
        return best;
    }
    b200_ndt* handle() { sync(); return ndt_; }

   private:
    void sync() {
        if (!ndt_ || dirty_) {
            if (ndt_) b200_ndt_destroy(ndt_);
            ndt_ = nullptr;
            check(b200_ndt_create(&prm_, device_, &ndt_), "b200_ndt_create");
            dirty_ = false;
            target_dirty_ = target_ != nullptr;
            source_dirty_ = source_ != nullptr;
        }
        using PointT = typename std::remove_reference<decltype(target_->points[0])>::type;
        if (target_dirty_ && target_) {
            check(b200_ndt_set_target(ndt_, reinterpret_cast<const float*>(target_->points.data()), (int64_t)target_->points.size(), sizeof(PointT)),
                  "b200_ndt_set_target");
            target_dirty_ = false;
        }
        if (source_dirty_ && source_) {
            check(b200_ndt_set_source(ndt_, reinterpret_cast<const float*>(source_->points.data()), (int64_t)source_->points.size(), sizeof(PointT)),
                  "b200_ndt_set_source");
            source_dirty_ = false;
        }
    }
    int device_;
    b200_ndt_params prm_{};
    b200_ndt* ndt_ = nullptr;
    bool dirty_ = true, target_dirty_ = false, source_dirty_ = false;
    std::shared_ptr<const CloudT> target_, source_;
    float final_[16];
    b200_ndt_result result_{};
};

/// Batched loop-closure registration (b200_ndt_pairs_align): P independent (source, target, guess) pairs in one call, each
/// exactly what a fresh pclomp NDT with these settings would compute for it alone.  A batched performLoopClosure thread or
/// an offline loop-verification tool fills the candidate lists and reads hasConverged(p) / getFitnessScore(p) /
/// getFinalTransformation(p), the three quantities mapOptmization.cpp:683-693 gates on.
template <typename CloudT>
class NdtPairBatch {
   public:
    explicit NdtPairBatch(int device = 0) : device_(device) {
        prm_.resolution = 1.0f; prm_.step_size = 0.1; prm_.outlier_ratio = 0.55; prm_.trans_eps = 0.1;
        prm_.max_iter = 35; prm_.search = 7; prm_.min_pts = 6; prm_.eig_ratio = 0.01;
    }
    ~NdtPairBatch() { b200_ndt_pairs_destroy(h_); }
    NdtPairBatch(const NdtPairBatch&) = delete;
    NdtPairBatch& operator=(const NdtPairBatch&) = delete;

    void setResolution(float r) { prm_.resolution = r; dirty_ = true; }
    void setStepSize(double s) { prm_.step_size = s; dirty_ = true; }
    void setOutlierRatio(double o) { prm_.outlier_ratio = o; dirty_ = true; }
    void setTransformationEpsilon(double e) { prm_.trans_eps = e; dirty_ = true; }
    void setMaximumIterations(int n) { prm_.max_iter = n; dirty_ = true; }
    void setNumThreads(int) {}
    void setNeighborhoodSearchMethod(NeighborSearchMethod m) {
        prm_.search = m == KDTREE ? 0 : m == DIRECT1 ? 1 : m == DIRECT26 ? 27 : 7;
        dirty_ = true;
    }

    /// sources[p] / targets[p] = pair p; guesses16 = P x 16 column-major (NULL = identity, as the reference calls it);
    /// max_range = the getFitnessScore argument.  Per-pair failures (an empty cloud, a target without a finite point) are in
    /// status(p); a malformed call throws.
    void align(const std::vector<const CloudT*>& sources, const std::vector<const CloudT*>& targets, const float* guesses16 = nullptr,
               double max_range = 1.7976931348623157e308) {
        if (sources.size() != targets.size() || sources.empty()) throw std::runtime_error("NdtPairBatch::align: one target per source, at least one pair");
        ensure();
        const size_t P = sources.size();
        std::vector<int64_t> soff(P + 1, 0), toff(P + 1, 0);
        for (size_t p = 0; p < P; ++p) {
            soff[p + 1] = soff[p] + (int64_t)sources[p]->points.size();
            toff[p + 1] = toff[p] + (int64_t)targets[p]->points.size();
        }
        src_.resize(3 * (size_t)std::max<int64_t>(soff[P], 1));
        tgt_.resize(3 * (size_t)std::max<int64_t>(toff[P], 1));
        for (size_t p = 0; p < P; ++p) {
            float* s = src_.data() + 3 * soff[p];
            for (const auto& q : sources[p]->points) { *s++ = q.x; *s++ = q.y; *s++ = q.z; }
            float* t = tgt_.data() + 3 * toff[p];
            for (const auto& q : targets[p]->points) { *t++ = q.x; *t++ = q.y; *t++ = q.z; }
        }
        res_.assign(P, b200_ndt_pair_result{});
        check(b200_ndt_pairs_align(nullptr, h_, src_.data(), soff.data(), tgt_.data(), toff.data(), 12, (int64_t)P, guesses16, max_range, res_.data()),
              "b200_ndt_pairs_align");
    }
    /// performLoopClosure up to the fitness gate for the query keyframes cur (mapOptmization.cpp: detectLoopClosureDistance or
    /// detectLoopClosureExternal, loopFindNearKeyframes for both sides, the 300 / 1000 size gates, align(identity),
    /// getFitnessScore(max_range)), all on the device: pre empty = detect by distance, otherwise pre[q] is query q's partner
    /// (-1 = none).  Query q's record is then result(q) / hasConverged(q) / getFitnessScore(q) / getFinalTransformation(q);
    /// loopResult(q) adds the partner and the downsampled sizes.  status(q) == B200_NO_EFFECTIVE_POINTS: not registered.
    template <class KeyframesT>
    void closeLoops(KeyframesT& store, const std::vector<int64_t>& cur, const std::vector<int64_t>& pre, const b200_loop_params& prm) {
        if (cur.empty() || (!pre.empty() && pre.size() != cur.size())) throw std::runtime_error("NdtPairBatch::closeLoops: one partner per query, at least one query");
        ensure();
        loop_.assign(cur.size(), b200_loop_result{});
        check(b200_loop_close(nullptr, h_, store.handle(), cur.data(), pre.empty() ? nullptr : pre.data(), (int64_t)cur.size(), &prm, loop_.data()),
              "b200_loop_close");
        res_.resize(cur.size());
        for (size_t q = 0; q < cur.size(); ++q) res_[q] = loop_[q].reg;
    }
    const b200_loop_result& loopResult(size_t q) const { return loop_.at(q); }
    size_t size() const { return res_.size(); }
    int status(size_t p) const { return res_.at(p).status; }
    bool hasConverged(size_t p) const { return res_.at(p).status == B200_OK && res_[p].ndt.converged != 0; }
    const float* getFinalTransformation(size_t p) const { return res_.at(p).final16; }   // column-major 4x4
    double getFitnessScore(size_t p) const { return res_.at(p).fitness; }
    int getFinalNumIteration(size_t p) const { return res_.at(p).ndt.iters; }
    double getTransformationProbability(size_t p) const { return res_.at(p).ndt.trans_probability; }
    const b200_ndt_pair_result& result(size_t p) const { return res_.at(p); }

   private:
    void ensure() {
        if (!h_ || dirty_) {
            if (h_) b200_ndt_pairs_destroy(h_);
            h_ = nullptr;
            check(b200_ndt_pairs_create(&prm_, device_, &h_), "b200_ndt_pairs_create");
            dirty_ = false;
        }
    }
    int device_;
    b200_ndt_params prm_{};
    b200_ndt_pairs* h_ = nullptr;
    bool dirty_ = true;
    std::vector<float> src_, tgt_;
    std::vector<b200_ndt_pair_result> res_;
    std::vector<b200_loop_result> loop_;
};

/// The keyframes of a session on the device: cornerCloudKeyFrames / surfCloudKeyFrames / cloudKeyPoses6D of mapOptmization.cpp.
/// add() stores the corner cloud followed by the surf cloud (the order loopFindNearKeyframes appends them in) with the
/// keyframe's pose {x, y, z, roll, pitch, yaw} and time; setPoses() is correctPoses() after a graph optimisation.
template <class CloudT>
class KeyframeStore {
   public:
    explicit KeyframeStore(int device = 0) { check(b200_keyframes_create(device, &h_), "b200_keyframes_create"); }
    ~KeyframeStore() { b200_keyframes_destroy(h_); }
    KeyframeStore(const KeyframeStore&) = delete;
    KeyframeStore& operator=(const KeyframeStore&) = delete;

    /// the corner / surf split is kept for ScanToMap::extractSurroundingKeyFrames (b200_keyframes_add_features)
    int64_t add(const CloudT& corner, const CloudT& surf, const float pose6[6], double time) {
        xyzi_.clear();
        for (const CloudT* c : {&corner, &surf})
            for (const auto& q : c->points) { xyzi_.push_back(q.x); xyzi_.push_back(q.y); xyzi_.push_back(q.z); xyzi_.push_back(q.intensity); }
        const int64_t nc = (int64_t)corner.points.size(), ns = (int64_t)surf.points.size();
        int64_t key = -1;
        check(b200_keyframes_add_features(h_, nc ? xyzi_.data() : nullptr, nc, 16, ns ? xyzi_.data() + 4 * nc : nullptr, ns, 16, pose6, time, &key),
              "b200_keyframes_add_features");
        return key;
    }
    /// the same from clouds on the device (b200host::FeatureExtraction::deviceCloud, float4 records)
    int64_t add(const void* d_corner, int64_t n_corner, const void* d_surf, int64_t n_surf, const float pose6[6], double time) {
        int64_t key = -1;
        check(b200_keyframes_add_features_device(h_, d_corner, n_corner, d_surf, n_surf, pose6, time, &key), "b200_keyframes_add_features_device");
        return key;
    }
    void setPoses(int64_t first, int64_t count, const float* poses6) { check(b200_keyframes_set_poses(h_, first, count, poses6), "b200_keyframes_set_poses"); }
    int64_t size() const { return b200_keyframes_count(h_); }
    /// detectLoopClosureDistance for the query keyframes cur: pre[q] = -1 without a candidate
    std::vector<int64_t> detect(const std::vector<int64_t>& cur, const b200_loop_params& prm) {
        std::vector<int64_t> pre(cur.size(), -1);
        if (!cur.empty()) check(b200_loop_detect(h_, cur.data(), (int64_t)cur.size(), &prm, pre.data(), nullptr), "b200_loop_detect");
        return pre;
    }
    b200_keyframes* handle() { return h_; }

   private:
    b200_keyframes* h_ = nullptr;
    std::vector<float> xyzi_;
};

}  // namespace b200host
