// cupoch_b200_facade.h -- header-only C++17 facade that reproduces the cupoch
// classes on the ICP / kNN / voxel-grid path on top of the C ABI
// (include/cupoch_b200.h).  Names, argument meaning and error behaviour follow
// the reference headers cited at each declaration; no thrust, no CUDA headers.
//
// Eigen: used when available (cupoch's API types are Eigen's); otherwise
// layout-compatible PODs are declared in namespace Eigen so that the facade
// still builds where Eigen is absent (it is absent in the build container).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <tuple>
#include <utility>
#include <limits>
#include <vector>

#include "cupoch_b200.h"

#if __has_include(<Eigen/Core>)
#include <Eigen/Core>
namespace Eigen {
typedef Matrix<float, 4, 4, DontAlign> Matrix4f_u;
}
#else
namespace Eigen {
struct Vector3f {
    float v[3];
    Vector3f() : v{0, 0, 0} {}
    Vector3f(float x, float y, float z) : v{x, y, z} {}
    float &operator[](int i) { return v[i]; }
    float operator[](int i) const { return v[i]; }
    float &operator()(int i) { return v[i]; }
    float operator()(int i) const { return v[i]; }
    static Vector3f Zero() { return Vector3f(); }
};
struct Vector3i {
    int v[3];
    Vector3i() : v{0, 0, 0} {}
    Vector3i(int a, int b, int c) : v{a, b, c} {}
    int &operator[](int i) { return v[i]; }
    int operator[](int i) const { return v[i]; }
    int &operator()(int i) { return v[i]; }
    int operator()(int i) const { return v[i]; }
};
struct Vector2i {
    int v[2];
    Vector2i() : v{0, 0} {}
    Vector2i(int a, int b) : v{a, b} {}
    int &operator[](int i) { return v[i]; }
    int operator[](int i) const { return v[i]; }
};
struct Matrix3f {  // column-major like Eigen's default
    float m[9];
    Matrix3f() : m{0, 0, 0, 0, 0, 0, 0, 0, 0} {}
    float &operator()(int r, int c) { return m[3 * c + r]; }
    float operator()(int r, int c) const { return m[3 * c + r]; }
};
struct Matrix4f {  // column-major
    float m[16];
    Matrix4f() { std::memset(m, 0, sizeof(m)); }
    float &operator()(int r, int c) { return m[4 * c + r]; }
    float operator()(int r, int c) const { return m[4 * c + r]; }
    static Matrix4f Identity() {
        Matrix4f I;
        for (int i = 0; i < 4; ++i) I(i, i) = 1.f;
        return I;
    }
    bool isIdentity(float prec = 1e-5f) const {
        for (int r = 0; r < 4; ++r)
            for (int c = 0; c < 4; ++c)
                if (std::fabs((*this)(r, c) - (r == c ? 1.f : 0.f)) > prec) return false;
        return true;
    }
    Matrix4f operator*(const Matrix4f &o) const {
        Matrix4f R;
        for (int r = 0; r < 4; ++r)
            for (int c = 0; c < 4; ++c)
                R(r, c) = (((*this)(r, 0) * o(0, c) + (*this)(r, 1) * o(1, c)) + (*this)(r, 2) * o(2, c)) + (*this)(r, 3) * o(3, c);
        return R;
    }
};
typedef Matrix4f Matrix4f_u;
}  // namespace Eigen
#endif

namespace cupoch {
namespace utility {

inline void LogError(const char *msg) { std::fprintf(stderr, "[cupoch_b200][error] %s\n", msg); }
inline void LogWarning(const char *msg) { std::fprintf(stderr, "[cupoch_b200][warning] %s\n", msg); }
inline void check(int rc) {
    if (rc != CPHB_OK) throw std::runtime_error(std::string("cupoch_b200: ") + cphb_last_error());
}

/// RAII device array (stands in for rmm/thrust device_vector, device_vector.h:67-105).
template <typename T>
class device_vector {
public:
    device_vector() {}
    explicit device_vector(size_t n) { resize(n); }
    device_vector(const std::vector<T> &h) { *this = h; }
    device_vector(const device_vector &o) { copy_from(o); }
    device_vector(device_vector &&o) noexcept : p_(o.p_), n_(o.n_), cap_(o.cap_) { o.p_ = nullptr; o.n_ = o.cap_ = 0; }
    ~device_vector() { cphb_free(p_); }
    device_vector &operator=(const device_vector &o) { if (this != &o) copy_from(o); return *this; }
    device_vector &operator=(device_vector &&o) noexcept {
        if (this != &o) { cphb_free(p_); p_ = o.p_; n_ = o.n_; cap_ = o.cap_; o.p_ = nullptr; o.n_ = o.cap_ = 0; }
        return *this;
    }
    device_vector &operator=(const std::vector<T> &h) {
        resize(h.size());
        if (n_) { check(cphb_memcpy_h2d(p_, h.data(), n_ * sizeof(T), nullptr)); check(cphb_stream_synchronize(nullptr)); }
        return *this;
    }
    void resize(size_t n) {
        if (n > cap_) {
            T *q = static_cast<T *>(cphb_malloc(n * sizeof(T)));
            if (!q) check(CPHB_ERR_CUDA);
            if (n_) check(cphb_memcpy_d2d(q, p_, n_ * sizeof(T), nullptr));
            check(cphb_stream_synchronize(nullptr));
            cphb_free(p_);
            p_ = q;
            cap_ = n;
        }
        n_ = n;
    }
    void clear() { n_ = 0; }
    size_t size() const { return n_; }
    bool empty() const { return n_ == 0; }
    T *data() { return p_; }
    const T *data() const { return p_; }
    std::vector<T> to_host() const {
        std::vector<T> h(n_);
        if (n_) { check(cphb_memcpy_d2h(h.data(), p_, n_ * sizeof(T), nullptr)); check(cphb_stream_synchronize(nullptr)); }
        return h;
    }

private:
    void copy_from(const device_vector &o) {
        resize(o.n_);
        if (n_) { check(cphb_memcpy_d2d(p_, o.p_, n_ * sizeof(T), nullptr)); check(cphb_stream_synchronize(nullptr)); }
    }
    T *p_ = nullptr;
    size_t n_ = 0, cap_ = 0;
};

inline void to_row_major(const Eigen::Matrix4f &M, float out[16]) {
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) out[4 * r + c] = M(r, c);
}
inline Eigen::Matrix4f from_row_major(const float in[16]) {
    Eigen::Matrix4f M;
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) M(r, c) = in[4 * r + c];
    return M;
}
}  // namespace utility

// --------------------------------------------------------------------------- knn
namespace knn {
static const int NUM_MAX_NN = 100;  // kdtree_search_param.h:26

class KDTreeSearchParam {  // kdtree_search_param.h:28-66
public:
    enum class SearchType { Knn = 0, Radius = 1 };
    virtual ~KDTreeSearchParam() {}
    SearchType GetSearchType() const { return search_type_; }

protected:
    KDTreeSearchParam(SearchType t) : search_type_(t) {}

private:
    SearchType search_type_;
};
class KDTreeSearchParamKNN : public KDTreeSearchParam {
public:
    KDTreeSearchParamKNN(int knn = 30) : KDTreeSearchParam(SearchType::Knn), knn_(knn) {}
    int knn_;
};
class KDTreeSearchParamRadius : public KDTreeSearchParam {
public:
    KDTreeSearchParamRadius(float radius, int max_nn) : KDTreeSearchParam(SearchType::Radius), radius_(radius), max_nn_(max_nn) {}
    float radius_;
    int max_nn_;
};

/// knn::KDTreeFlann (kdtree_flann.h:43-124).  Non-copyable; copies the data like the reference.
class KDTreeFlann {
public:
    KDTreeFlann() {}
    KDTreeFlann(const utility::device_vector<Eigen::Vector3f> &data) { SetRawData(data); }
    ~KDTreeFlann() { release(); }
    KDTreeFlann(const KDTreeFlann &) = delete;
    KDTreeFlann &operator=(const KDTreeFlann &) = delete;

    bool SetRawData(const utility::device_vector<Eigen::Vector3f> &data) {
        release();
        n_ = data.size();
        if (n_ == 0) return false;  // kdtree_flann.inl:128-131
        utility::check(cphb_index_create(reinterpret_cast<const float *>(data.data()), n_, nullptr, &ix_));
        return true;
    }
    int Search(const utility::device_vector<Eigen::Vector3f> &query, const KDTreeSearchParam &param,
               utility::device_vector<int> &indices, utility::device_vector<float> &distance2) const {
        switch (param.GetSearchType()) {
            case KDTreeSearchParam::SearchType::Knn:
                return SearchKNN(query, static_cast<const KDTreeSearchParamKNN &>(param).knn_, indices, distance2);
            case KDTreeSearchParam::SearchType::Radius: {
                const auto &p = static_cast<const KDTreeSearchParamRadius &>(param);
                return SearchRadius(query, p.radius_, p.max_nn_, indices, distance2);
            }
        }
        return -1;
    }
    int SearchKNN(const utility::device_vector<Eigen::Vector3f> &query, int knn, utility::device_vector<int> &indices,
                  utility::device_vector<float> &distance2) const {
        if (!ix_ || n_ == 0 || query.empty() || knn < 0 || knn > NUM_MAX_NN) return -1;  // kdtree_flann.cu:46-48
        indices.resize(query.size() * knn);
        distance2.resize(query.size() * knn);
        int64_t cnt = 0;
        int rc = cphb_search_knn(ix_, reinterpret_cast<const float *>(query.data()), query.size(), knn, indices.data(),
                                 distance2.data(), &cnt, nullptr);
        return rc == CPHB_OK ? (int)cnt : -1;
    }
    int SearchRadius(const utility::device_vector<Eigen::Vector3f> &query, float radius, int max_nn,
                     utility::device_vector<int> &indices, utility::device_vector<float> &distance2) const {
        if (!ix_ || n_ == 0 || query.empty() || max_nn < 0) return -1;  // kdtree_flann.cu:70-72
        indices.resize(query.size() * max_nn);
        distance2.resize(query.size() * max_nn);
        int64_t cnt = 0;
        int rc = cphb_search_radius(ix_, reinterpret_cast<const float *>(query.data()), query.size(), radius, max_nn,
                                    indices.data(), distance2.data(), &cnt, nullptr);
        return rc == CPHB_OK ? (int)cnt : -1;
    }
    /// north_star's name for SearchRadius (SURVEY.md section 0).
    int SearchHybrid(const utility::device_vector<Eigen::Vector3f> &query, float radius, int max_nn,
                     utility::device_vector<int> &indices, utility::device_vector<float> &distance2) const {
        return SearchRadius(query, radius, max_nn, indices, distance2);
    }
    // single host query overloads (kdtree_flann.cu:88-129)
    int SearchKNN(const Eigen::Vector3f &query, int knn, std::vector<int> &indices, std::vector<float> &distance2) const {
        utility::device_vector<Eigen::Vector3f> q(std::vector<Eigen::Vector3f>{query});
        utility::device_vector<int> i;
        utility::device_vector<float> d;
        int k = SearchKNN(q, knn, i, d);
        indices = i.to_host();
        distance2 = d.to_host();
        return k;
    }
    int SearchRadius(const Eigen::Vector3f &query, float radius, int max_nn, std::vector<int> &indices,
                     std::vector<float> &distance2) const {
        utility::device_vector<Eigen::Vector3f> q(std::vector<Eigen::Vector3f>{query});
        utility::device_vector<int> i;
        utility::device_vector<float> d;
        int k = SearchRadius(q, radius, max_nn, i, d);
        indices = i.to_host();
        distance2 = d.to_host();
        return k;
    }

private:
    void release() {
        if (ix_) { cphb_stream_synchronize(nullptr); cphb_index_destroy(ix_); ix_ = nullptr; }
    }
    cphb_index *ix_ = nullptr;
    size_t n_ = 0;
};
}  // namespace knn

// --------------------------------------------------------------------------- geometry
namespace geometry {
/// geometry::PointCloud (pointcloud.h:43-263), hot-path subset.
class PointCloud {
public:
    PointCloud() {}
    PointCloud(const std::vector<Eigen::Vector3f> &points) : points_(points) {}
    virtual ~PointCloud() {}
    bool IsEmpty() const { return points_.empty(); }
    bool HasPoints() const { return !points_.empty(); }
    bool HasNormals() const { return !points_.empty() && normals_.size() == points_.size(); }          // pointcloud.h:82-94
    bool HasColors() const { return !points_.empty() && colors_.size() == points_.size(); }
    bool HasCovariances() const { return !points_.empty() && covariances_.size() == points_.size(); }
    void SetPoints(const std::vector<Eigen::Vector3f> &p) { points_ = p; }
    void SetNormals(const std::vector<Eigen::Vector3f> &p) { normals_ = p; }
    void SetColors(const std::vector<Eigen::Vector3f> &p) { colors_ = p; }
    std::vector<Eigen::Vector3f> GetPoints() const { return points_.to_host(); }
    std::vector<Eigen::Vector3f> GetNormals() const { return normals_.to_host(); }
    std::vector<Eigen::Vector3f> GetColors() const { return colors_.to_host(); }

    Eigen::Vector3f GetMinBound() const { return bound(0); }  // pointcloud.cu:205
    Eigen::Vector3f GetMaxBound() const { return bound(1); }

    PointCloud &Transform(const Eigen::Matrix4f &T) {  // pointcloud.cu:293-299
        float t[16];
        utility::to_row_major(T, t);
        if (!points_.empty())
            utility::check(cphb_transform(fp(points_), HasNormals() ? fp(normals_) : nullptr,
                                          HasCovariances() ? fp(covariances_) : nullptr, 1, points_.size(), t, nullptr));
        utility::check(cphb_stream_synchronize(nullptr));
        return *this;
    }
    std::shared_ptr<PointCloud> VoxelDownSample(float voxel_size) const {  // down_sample.cu:170-273
        auto out = std::make_shared<PointCloud>();
        if (voxel_size <= 0.0) { utility::LogWarning("[VoxelDownSample] voxel_size <= 0."); return out; }
        const size_t n = points_.size();
        if (n == 0) return out;
        const bool hn = HasNormals(), hc = HasColors();
        out->points_.resize(n);
        if (hn) out->normals_.resize(n);
        if (hc) out->colors_.resize(n);
        size_t m = 0;
        utility::check(cphb_voxel_down_sample(cfp(points_), hn ? cfp(normals_) : nullptr, hc ? cfp(colors_) : nullptr, n,
                                              voxel_size, fp(out->points_), hn ? fp(out->normals_) : nullptr,
                                              hc ? fp(out->colors_) : nullptr, &m, nullptr));
        out->points_.resize(m);
        if (hn) out->normals_.resize(m);
        if (hc) out->colors_.resize(m);
        return out;
    }
    bool EstimateNormals(const knn::KDTreeSearchParam &param = knn::KDTreeSearchParamKNN()) {  // estimate_normals.cu:82-127
        if (!HasNormals()) normals_.resize(points_.size());
        int knn = 0, max_nn = 0;
        float radius = 0.f;
        if (param.GetSearchType() == knn::KDTreeSearchParam::SearchType::Knn) knn = static_cast<const knn::KDTreeSearchParamKNN &>(param).knn_;
        else { radius = static_cast<const knn::KDTreeSearchParamRadius &>(param).radius_; max_nn = static_cast<const knn::KDTreeSearchParamRadius &>(param).max_nn_; }
        utility::check(cphb_estimate_normals(cfp(points_), points_.size(), knn, radius, max_nn, fp(normals_), nullptr));
        return true;
    }
    /// PointCloud::SelectByIndex (down_sample.cu:110-127).  Index vectors are size_t like the reference's.
    std::shared_ptr<PointCloud> SelectByIndex(const utility::device_vector<size_t> &indices, bool invert = false) const {
        std::vector<size_t> h = indices.to_host();
        const size_t n = points_.size();
        std::vector<int32_t> sel;
        if (invert) {  // sort + set_difference(0..n, indices) there: ascending complement
            std::vector<char> drop(n, 0);
            for (size_t i : h) if (i < n) drop[i] = 1;
            for (size_t i = 0; i < n; ++i) if (!drop[i]) sel.push_back((int32_t)i);
        } else {
            sel.reserve(h.size());
            for (size_t i : h) sel.push_back((int32_t)i);
        }
        utility::device_vector<int32_t> d;
        d = sel;
        return gather(d, sel.size());
    }
    /// PointCloud::RemoveRadiusOutliers (down_sample.cu:317-354) -> (filtered cloud, kept indices)
    std::tuple<std::shared_ptr<PointCloud>, utility::device_vector<size_t>> RemoveRadiusOutliers(size_t nb_points,
                                                                                                   float search_radius) const {
        if (nb_points < 1 || search_radius <= 0)
            utility::LogError("[RemoveRadiusOutliers] Illegal input parameters, number of points and radius must be positive");
        utility::device_vector<int32_t> kept(points_.size());
        size_t m = 0;
        if (!points_.empty())
            utility::check(cphb_remove_radius_outliers(cfp(points_), points_.size(), (int)nb_points, search_radius, kept.data(), &m,
                                                       nullptr));
        return finish_filter(kept, m);
    }
    /// PointCloud::RemoveStatisticalOutliers (down_sample.cu:356-438) -> (filtered cloud, kept indices)
    std::tuple<std::shared_ptr<PointCloud>, utility::device_vector<size_t>> RemoveStatisticalOutliers(size_t nb_neighbors,
                                                                                                        float std_ratio) const {
        if (nb_neighbors < 1 || std_ratio <= 0)
            utility::LogError("[RemoveStatisticalOutliers] Illegal input parameters, number of neighbors and standard deviation "
                              "ratio must be positive");
        utility::device_vector<int32_t> kept(points_.size());
        size_t m = 0;
        if (!points_.empty())
            utility::check(cphb_remove_statistical_outliers(cfp(points_), points_.size(), (int)nb_neighbors, std_ratio, kept.data(),
                                                            &m, nullptr, nullptr));
        return finish_filter(kept, m);
    }
    /// PointCloud::ClusterDBSCAN (pointcloud.h:195-199, pointcloud_cluster.cu:84-179): labels, -1 = noise
    std::unique_ptr<utility::device_vector<int>> ClusterDBSCAN(float eps, size_t min_points, bool print_progress = false,
                                                               size_t max_edges = 100) const {
        (void)print_progress;
        auto labels = std::make_unique<utility::device_vector<int>>(points_.size());
        if (!points_.empty())
            utility::check(cphb_cluster_dbscan(cfp(points_), points_.size(), eps, (int)min_points, (int)max_edges,
                                               reinterpret_cast<int32_t *>(labels->data()), nullptr, nullptr));
        return labels;
    }
    /// PointCloud::GaussianFilter (pointcloud.cu:387-433)
    std::shared_ptr<PointCloud> GaussianFilter(float search_radius, float sigma2, size_t num_max_search_points = 50) const {
        auto out = std::make_shared<PointCloud>();
        if (search_radius <= 0 || sigma2 <= 0 || num_max_search_points <= 0) {
            utility::LogError("[GaussianFilter] Illegal input parameters, radius and sigma2 must be positive.");
            return out;
        }
        const size_t n = points_.size();
        if (n == 0) return out;
        const bool hn = HasNormals(), hc = HasColors();
        out->points_.resize(n);
        if (hn) out->normals_.resize(n);
        if (hc) out->colors_.resize(n);
        size_t m = 0;
        utility::check(cphb_gaussian_filter(cfp(points_), hn ? cfp(normals_) : nullptr, hc ? cfp(colors_) : nullptr, n, search_radius,
                                            sigma2, (int)num_max_search_points, fp(out->points_), hn ? fp(out->normals_) : nullptr,
                                            hc ? fp(out->colors_) : nullptr, &m, nullptr));
        return out;
    }
    cphb_cloud view() const {
        cphb_cloud c;
        std::memset(&c, 0, sizeof(c));
        c.points = cfp(points_);
        c.n = points_.size();
        c.normals = HasNormals() ? cfp(normals_) : nullptr;
        c.colors = HasColors() ? cfp(colors_) : nullptr;
        c.covariances = HasCovariances() ? cfp(covariances_) : nullptr;
        c.color_gradient = (!points_.empty() && color_gradient_.size() == points_.size()) ? cfp(color_gradient_) : nullptr;
        c.cov_col_major = 1;  // Eigen::Matrix3f default storage
        return c;
    }

public:
    utility::device_vector<Eigen::Vector3f> points_, normals_, colors_;
    utility::device_vector<Eigen::Matrix3f> covariances_;
    utility::device_vector<Eigen::Vector3f> color_gradient_;  // PointCloudForColoredICP (colored_icp.cu:36-40)

private:
    template <class V> static float *fp(V &v) { return reinterpret_cast<float *>(v.data()); }
    template <class V> static const float *cfp(const V &v) { return reinterpret_cast<const float *>(v.data()); }
    std::shared_ptr<PointCloud> gather(const utility::device_vector<int32_t> &idx, size_t m) const {
        auto out = std::make_shared<PointCloud>();
        if (m == 0 || points_.empty()) return out;
        const bool hn = HasNormals(), hc = HasColors();
        out->points_.resize(m);
        if (hn) out->normals_.resize(m);
        if (hc) out->colors_.resize(m);
        utility::check(cphb_select_by_index(cfp(points_), hn ? cfp(normals_) : nullptr, hc ? cfp(colors_) : nullptr, points_.size(),
                                            idx.data(), m, fp(out->points_), hn ? fp(out->normals_) : nullptr,
                                            hc ? fp(out->colors_) : nullptr, nullptr));
        utility::check(cphb_stream_synchronize(nullptr));
        return out;
    }
    std::tuple<std::shared_ptr<PointCloud>, utility::device_vector<size_t>> finish_filter(utility::device_vector<int32_t> &kept,
                                                                                            size_t m) const {
        auto out = gather(kept, m);
        kept.resize(m);
        std::vector<int32_t> h32 = kept.to_host();
        std::vector<size_t> h(h32.begin(), h32.end());  // the reference hands back device_vector<size_t>
        utility::device_vector<size_t> idx;
        idx = h;
        return std::make_tuple(out, std::move(idx));
    }
    Eigen::Vector3f bound(int which) const {
        float mn[3] = {0, 0, 0}, mx[3] = {0, 0, 0};
        if (!points_.empty()) utility::check(cphb_min_max_bound(cfp(points_), points_.size(), mn, mx, nullptr));
        return which ? Eigen::Vector3f(mx[0], mx[1], mx[2]) : Eigen::Vector3f(mn[0], mn[1], mn[2]);
    }
};

/// geometry::Voxel (voxelgrid.h:48-62)
class Voxel {
public:
    Voxel() {}
    Voxel(const Eigen::Vector3i &grid_index) : grid_index_(grid_index) {}
    Voxel(const Eigen::Vector3i &grid_index, const Eigen::Vector3f &color) : grid_index_(grid_index), color_(color) {}
    Eigen::Vector3i grid_index_ = Eigen::Vector3i(0, 0, 0);
    Eigen::Vector3f color_ = Eigen::Vector3f(1.0f, 1.0f, 1.0f);
};

/// geometry::VoxelGrid (voxelgrid.h:84-160): creation from a point cloud (voxelgrid_factory.cu:164-228) and the
/// accessors that need nothing else.  Keys and colours are kept as two device vectors (the reference zips keys
/// with Voxel{grid_index, color}); GetVoxels() hands back the reference's pair.
class VoxelGrid {
public:
    bool HasVoxels() const { return voxels_keys_.size() > 0; }
    bool HasColors() const { return true; }  // voxelgrid.h:112-114
    bool IsEmpty() const { return !HasVoxels(); }
    std::pair<std::vector<Eigen::Vector3i>, std::vector<Voxel>> GetVoxels() const {
        std::vector<Eigen::Vector3i> k = voxels_keys_.to_host();
        std::vector<Eigen::Vector3f> c = voxels_colors_.to_host();
        std::vector<Voxel> v(k.size());
        for (size_t i = 0; i < k.size(); ++i) v[i] = Voxel(k[i], c[i]);
        return std::make_pair(std::move(k), std::move(v));
    }
    Eigen::Vector3i GetVoxel(const Eigen::Vector3f &point) const {  // voxelgrid.cu:338-341
        return Eigen::Vector3i((int)std::floor((point[0] - origin_[0]) / voxel_size_), (int)std::floor((point[1] - origin_[1]) / voxel_size_),
                               (int)std::floor((point[2] - origin_[2]) / voxel_size_));
    }
    static std::shared_ptr<VoxelGrid> CreateFromPointCloudWithinBounds(const PointCloud &input, float voxel_size,
                                                                       const Eigen::Vector3f &min_bound,
                                                                       const Eigen::Vector3f &max_bound) {
        auto out = std::make_shared<VoxelGrid>();
        if (voxel_size <= 0.0) utility::LogError("[VoxelGridFromPointCloud] voxel_size <= 0.");
        out->voxel_size_ = voxel_size;
        out->origin_ = min_bound;
        const size_t n = input.points_.size();
        if (n == 0) return out;
        const float mn[3] = {min_bound[0], min_bound[1], min_bound[2]}, mx[3] = {max_bound[0], max_bound[1], max_bound[2]};
        out->voxels_keys_.resize(n);
        out->voxels_colors_.resize(n);
        size_t m = 0;
        utility::check(cphb_voxel_grid_from_point_cloud(
                reinterpret_cast<const float *>(input.points_.data()),
                input.HasColors() ? reinterpret_cast<const float *>(input.colors_.data()) : nullptr, n, voxel_size, mn, mx,
                reinterpret_cast<int32_t *>(out->voxels_keys_.data()), reinterpret_cast<float *>(out->voxels_colors_.data()), &m,
                nullptr));
        out->voxels_keys_.resize(m);
        out->voxels_colors_.resize(m);
        return out;
    }
    static std::shared_ptr<VoxelGrid> CreateFromPointCloud(const PointCloud &input, float voxel_size) {  // :221-228
        const Eigen::Vector3f lo = input.GetMinBound(), hi = input.GetMaxBound();
        const float h = voxel_size * 0.5f;
        return CreateFromPointCloudWithinBounds(input, voxel_size, Eigen::Vector3f(lo[0] - h, lo[1] - h, lo[2] - h),
                                                Eigen::Vector3f(hi[0] + h, hi[1] + h, hi[2] + h));
    }

public:
    float voxel_size_ = 0.0f;
    Eigen::Vector3f origin_ = Eigen::Vector3f(0.f, 0.f, 0.f);
    utility::device_vector<Eigen::Vector3i> voxels_keys_;
    utility::device_vector<Eigen::Vector3f> voxels_colors_;
};

/// geometry::OccupancyVoxel (occupancygrid.h:33-72)
class OccupancyVoxel {
public:
    OccupancyVoxel() {}
    OccupancyVoxel(const Eigen::Vector3i &grid_index, float prob_log) : grid_index_(grid_index), prob_log_(prob_log) {}
    Eigen::Vector3i grid_index_ = Eigen::Vector3i(0, 0, 0);           // (Vector3ui16 in the reference)
    Eigen::Vector3f color_ = Eigen::Vector3f(0.0f, 0.0f, 1.0f);
    float prob_log_ = std::numeric_limits<float>::quiet_NaN();
};

/// geometry::OccupancyGrid (occupancygrid.h:74-147): dense log-odds grid; Insert ray-casts a scan into it.  The members
/// the reference exposes (voxel_size_, origin_, the probability parameters) are public here too and are handed to the
/// engine at every call.  Extract* return host vectors of voxels (the reference returns device vectors of its 24-byte
/// voxel struct; the engine stores 4.1 bytes per cell and materialises voxels on request).
class OccupancyGrid {
public:
    OccupancyGrid() : OccupancyGrid(0.05f, 512) {}
    OccupancyGrid(float voxel_size, size_t resolution = 512, const Eigen::Vector3f &origin = Eigen::Vector3f(0.f, 0.f, 0.f))
        : voxel_size_(voxel_size), resolution_(resolution), origin_(origin) {
        const float o[3] = {origin[0], origin[1], origin[2]};
        utility::check(cphb_occgrid_create(voxel_size, (int)resolution, o, nullptr, &h_));
    }
    ~OccupancyGrid() { cphb_stream_synchronize(nullptr); cphb_occgrid_destroy(h_); }
    OccupancyGrid(const OccupancyGrid &) = delete;
    OccupancyGrid &operator=(const OccupancyGrid &) = delete;

    OccupancyGrid &Clear() { utility::check(cphb_occgrid_clear(h_, nullptr)); return *this; }
    bool HasVoxels() const { return true; }
    bool HasColors() const { return true; }
    Eigen::Vector3f GetMinBound() const {  // occupancygrid.cu:317-322
        int32_t lo[3], hi[3];
        utility::check(cphb_occgrid_bounds(h_, lo, hi, nullptr));
        const int h = (int)resolution_ / 2;
        return Eigen::Vector3f((lo[0] - h) * voxel_size_ + origin_[0], (lo[1] - h) * voxel_size_ + origin_[1], (lo[2] - h) * voxel_size_ + origin_[2]);
    }
    Eigen::Vector3f GetMaxBound() const {  // occupancygrid.cu:324-333
        int32_t lo[3], hi[3];
        utility::check(cphb_occgrid_bounds(h_, lo, hi, nullptr));
        const int h = (int)resolution_ / 2 - 1;
        return Eigen::Vector3f((hi[0] - h) * voxel_size_ + origin_[0], (hi[1] - h) * voxel_size_ + origin_[1], (hi[2] - h) * voxel_size_ + origin_[2]);
    }
    std::tuple<bool, OccupancyVoxel> GetVoxel(const Eigen::Vector3f &point) const {  // occupancygrid.cu:351-356
        sync();
        const float p[3] = {point[0], point[1], point[2]};
        int known = 0, gi[3];
        float prob = 0.f;
        utility::check(cphb_occgrid_get_voxel(h_, p, &known, &prob, gi, nullptr));
        return std::make_tuple(known != 0, OccupancyVoxel(Eigen::Vector3i(gi[0], gi[1], gi[2]), prob));
    }
    bool IsOccupied(const Eigen::Vector3f &point) const {
        auto r = GetVoxel(point);
        return std::get<0>(r) && std::get<1>(r).prob_log_ > occ_prob_thres_log_;
    }
    bool IsUnknown(const Eigen::Vector3f &point) const { return !std::get<0>(GetVoxel(point)); }
    std::shared_ptr<std::vector<OccupancyVoxel>> ExtractKnownVoxels() const { return extract(0); }
    std::shared_ptr<std::vector<OccupancyVoxel>> ExtractFreeVoxels() const { return extract(1); }
    std::shared_ptr<std::vector<OccupancyVoxel>> ExtractOccupiedVoxels() const { return extract(2); }
    OccupancyGrid &SetFreeArea(const Eigen::Vector3f &min_bound, const Eigen::Vector3f &max_bound) {
        sync();
        const float lo[3] = {min_bound[0], min_bound[1], min_bound[2]}, hi[3] = {max_bound[0], max_bound[1], max_bound[2]};
        utility::check(cphb_occgrid_set_free_area(h_, lo, hi, nullptr));
        return *this;
    }
    OccupancyGrid &Insert(const utility::device_vector<Eigen::Vector3f> &points, const Eigen::Vector3f &viewpoint, float max_range = -1.0f) {
        sync();
        const float v[3] = {viewpoint[0], viewpoint[1], viewpoint[2]};
        if (points.size()) utility::check(cphb_occgrid_insert(h_, reinterpret_cast<const float *>(points.data()), points.size(), v, max_range, nullptr));
        return *this;
    }
    OccupancyGrid &Insert(const std::vector<Eigen::Vector3f> &points, const Eigen::Vector3f &viewpoint, float max_range = -1.0f) {
        return Insert(utility::device_vector<Eigen::Vector3f>(points), viewpoint, max_range);
    }
    OccupancyGrid &Insert(const PointCloud &pointcloud, const Eigen::Vector3f &viewpoint, float max_range = -1.0f) {
        return Insert(pointcloud.points_, viewpoint, max_range);
    }
    OccupancyGrid &AddVoxel(const Eigen::Vector3i &voxel, bool occupied = false) {  // occupancygrid.cu:554-577
        sync();
        const int32_t v[3] = {voxel[0], voxel[1], voxel[2]};
        if (cphb_occgrid_add_voxel(h_, v, occupied ? 1 : 0, nullptr) != CPHB_OK)
            utility::LogError("[OccupancyGrid] a provided voxeld is not occupancy grid range.");
        return *this;
    }
    OccupancyGrid &AddVoxels(const utility::device_vector<Eigen::Vector3i> &voxels, bool occupied = false) {
        sync();
        if (voxels.size()) utility::check(cphb_occgrid_add_voxels(h_, reinterpret_cast<const int32_t *>(voxels.data()), voxels.size(), occupied ? 1 : 0, nullptr));
        return *this;
    }

public:
    float voxel_size_ = 0.05f;
    size_t resolution_ = 512;
    Eigen::Vector3f origin_ = Eigen::Vector3f(0.f, 0.f, 0.f);
    float clamping_thres_min_ = -2.0f;
    float clamping_thres_max_ = 3.5f;
    float prob_hit_log_ = 0.85f;
    float prob_miss_log_ = -0.4f;
    float occ_prob_thres_log_ = 0.0f;
    bool visualize_free_area_ = true;

private:
    void sync() const {  // the public members are the source of truth, like the reference's
        const float o[3] = {origin_[0], origin_[1], origin_[2]};
        utility::check(cphb_occgrid_set_geometry(h_, voxel_size_, o));
        cphb_occgrid_params p = {clamping_thres_min_, clamping_thres_max_, prob_hit_log_, prob_miss_log_, occ_prob_thres_log_};
        utility::check(cphb_occgrid_set_params(h_, &p));
    }
    std::shared_ptr<std::vector<OccupancyVoxel>> extract(int which) const {
        sync();
        size_t m = 0;
        utility::check(cphb_occgrid_extract(h_, which, nullptr, nullptr, 0, &m, nullptr));
        auto out = std::make_shared<std::vector<OccupancyVoxel>>(m);
        if (!m) return out;
        utility::device_vector<Eigen::Vector3i> idx(m);
        utility::device_vector<float> pr(m);
        utility::check(cphb_occgrid_extract(h_, which, reinterpret_cast<int32_t *>(idx.data()), pr.data(), m, &m, nullptr));
        const auto hi = idx.to_host();
        const auto hp = pr.to_host();
        for (size_t i = 0; i < m; ++i) (*out)[i] = OccupancyVoxel(hi[i], hp[i]);
        return out;
    }
    cphb_occgrid *h_ = nullptr;
};
}  // namespace geometry

// --------------------------------------------------------------------------- registration
namespace registration {
typedef utility::device_vector<Eigen::Vector2i> CorrespondenceSet;  // transformation_estimation.h:36

enum class TransformationEstimationType {  // transformation_estimation.h:40-47
    Unspecified = 0, PointToPoint = 1, PointToPlane = 2, SymmetricMethod = 3, ColoredICP = 4, GeneralizedICP = 5,
};

class ICPConvergenceCriteria {  // registration.h:35-49
public:
    ICPConvergenceCriteria(float relative_fitness = 1e-6, float relative_rmse = 1e-6, int max_iteration = 30)
        : relative_fitness_(relative_fitness), relative_rmse_(relative_rmse), max_iteration_(max_iteration) {}
    float relative_fitness_, relative_rmse_;
    int max_iteration_;
};

class RegistrationResult {  // registration.h:51-67
public:
    RegistrationResult(const Eigen::Matrix4f &T = Eigen::Matrix4f::Identity()) : transformation_(T) {}
    std::vector<Eigen::Vector2i> GetCorrespondenceSet() const { return correspondence_set_.to_host(); }
    Eigen::Matrix4f_u transformation_;
    CorrespondenceSet correspondence_set_;
    float inlier_rmse_ = 0.0f;
    float fitness_ = 0.0f;
};

inline cphb_icp_params make_params(int est, float max_dist, const ICPConvergenceCriteria &c, float det_thresh, float lambda) {
    cphb_icp_params p;
    std::memset(&p, 0, sizeof(p));
    p.estimation = est;
    p.max_correspondence_distance = max_dist;
    p.relative_fitness = c.relative_fitness_;
    p.relative_rmse = c.relative_rmse_;
    p.max_iteration = c.max_iteration_;
    p.det_thresh = det_thresh;
    p.lambda_geometric = lambda;
    return p;
}

/// transformation_estimation.h:49-77.  User subclasses (Unspecified) run through the generic loop below.
class TransformationEstimation {
public:
    virtual ~TransformationEstimation() {}
    virtual TransformationEstimationType GetTransformationEstimationType() const = 0;
    virtual float ComputeRMSE(const geometry::PointCloud &source, const geometry::PointCloud &target, const CorrespondenceSet &corres) const = 0;
    virtual Eigen::Matrix4f ComputeTransformation(const geometry::PointCloud &source, const geometry::PointCloud &target, const CorrespondenceSet &corres) const = 0;
    virtual float det_thresh() const { return -1.f; }
    virtual float lambda_geometric() const { return 0.968f; }

protected:
    float rmse_impl(const geometry::PointCloud &s, const geometry::PointCloud &t, const CorrespondenceSet &c) const {
        cphb_cloud sc = s.view(), tc = t.view();
        cphb_icp_params p = make_params((int)GetTransformationEstimationType(), 0.f, ICPConvergenceCriteria(), det_thresh(), lambda_geometric());
        float r = 0.f;
        utility::check(cphb_compute_rmse(p.estimation, &sc, &tc, reinterpret_cast<const int32_t *>(c.data()), c.size(), &p, &r, nullptr));
        return r;
    }
    Eigen::Matrix4f transform_impl(const geometry::PointCloud &s, const geometry::PointCloud &t, const CorrespondenceSet &c) const {
        cphb_cloud sc = s.view(), tc = t.view();
        cphb_icp_params p = make_params((int)GetTransformationEstimationType(), 0.f, ICPConvergenceCriteria(), det_thresh(), lambda_geometric());
        float T[16];
        utility::check(cphb_compute_transformation(p.estimation, &sc, &tc, reinterpret_cast<const int32_t *>(c.data()), c.size(), &p, T, nullptr));
        return utility::from_row_major(T);
    }
};
#define CPHB_FACADE_ESTIMATOR_BODY(TYPE)                                                                        \
    TransformationEstimationType GetTransformationEstimationType() const override { return TransformationEstimationType::TYPE; } \
    float ComputeRMSE(const geometry::PointCloud &s, const geometry::PointCloud &t, const CorrespondenceSet &c) const override { return rmse_impl(s, t, c); } \
    Eigen::Matrix4f ComputeTransformation(const geometry::PointCloud &s, const geometry::PointCloud &t, const CorrespondenceSet &c) const override { return transform_impl(s, t, c); }

class TransformationEstimationPointToPoint : public TransformationEstimation {
public:
    CPHB_FACADE_ESTIMATOR_BODY(PointToPoint)
};
class TransformationEstimationPointToPlane : public TransformationEstimation {
public:
    TransformationEstimationPointToPlane(float det_thresh = 1.0e-6) : det_thresh_(det_thresh) {}
    CPHB_FACADE_ESTIMATOR_BODY(PointToPlane)
    float det_thresh() const override { return det_thresh_; }
    float det_thresh_;
};
class TransformationEstimationSymmetricMethod : public TransformationEstimation {
public:
    TransformationEstimationSymmetricMethod(float det_thresh = 1.0e-6) : det_thresh_(det_thresh) {}
    CPHB_FACADE_ESTIMATOR_BODY(SymmetricMethod)
    float det_thresh() const override { return det_thresh_; }
    float det_thresh_;
};
class TransformationEstimationForGeneralizedICP : public TransformationEstimation {  // generalized_icp.h:14-52
public:
    TransformationEstimationForGeneralizedICP(float epsilon = 1e-3) : epsilon_(epsilon) {}
    CPHB_FACADE_ESTIMATOR_BODY(GeneralizedICP)
    float epsilon_;
};
class TransformationEstimationForColoredICP : public TransformationEstimation {  // colored_icp.cu:42-71
public:
    TransformationEstimationForColoredICP(float lambda_geometric = 0.968, float det_thresh = 1.0e-6)
        : lambda_geometric_(lambda_geometric), det_thresh_(det_thresh) {
        if (lambda_geometric_ < 0 || lambda_geometric_ > 1.0) lambda_geometric_ = 0.968;
    }
    CPHB_FACADE_ESTIMATOR_BODY(ColoredICP)
    float det_thresh() const override { return det_thresh_; }
    float lambda_geometric() const override { return lambda_geometric_; }
    float lambda_geometric_, det_thresh_;
};

inline RegistrationResult to_result(const cphb_icp_result &r, CorrespondenceSet &&corr) {
    RegistrationResult out(utility::from_row_major(r.transformation));
    corr.resize((size_t)r.n_local_correspondences);
    out.correspondence_set_ = std::move(corr);
    out.fitness_ = r.fitness;
    out.inlier_rmse_ = r.inlier_rmse;
    return out;
}

/// registration::EvaluateRegistration (registration.cu:106-119)
inline RegistrationResult EvaluateRegistration(const geometry::PointCloud &source, const geometry::PointCloud &target,
                                               float max_correspondence_distance,
                                               const Eigen::Matrix4f &transformation = Eigen::Matrix4f::Identity()) {
    cphb_cloud sc = source.view(), tc = target.view();
    float T[16];
    utility::to_row_major(transformation, T);
    cphb_icp_result r;
    CorrespondenceSet corr(source.points_.size() ? source.points_.size() : 1);
    utility::check(cphb_evaluate_registration(&sc, &tc, max_correspondence_distance, T, &r, reinterpret_cast<int32_t *>(corr.data()), nullptr));
    return to_result(r, std::move(corr));
}

/// registration::RegistrationICP (registration.cu:121-173).  Built-in estimators run the fused
/// one-launch-per-iteration path; user-defined ones (Unspecified) the generic loop with the
/// caller's virtual ComputeTransformation, exactly as the reference's loop is written.
inline RegistrationResult RegistrationICP(const geometry::PointCloud &source, const geometry::PointCloud &target,
                                          float max_correspondence_distance,
                                          const Eigen::Matrix4f &init = Eigen::Matrix4f::Identity(),
                                          const TransformationEstimation &estimation = TransformationEstimationPointToPoint(),
                                          const ICPConvergenceCriteria &criteria = ICPConvergenceCriteria()) {
    if (max_correspondence_distance <= 0.0) utility::LogError("Invalid max_correspondence_distance.");  // :130-132
    const auto type = estimation.GetTransformationEstimationType();
    if ((type == TransformationEstimationType::PointToPlane || type == TransformationEstimationType::ColoredICP) && !target.HasNormals())
        utility::LogError("TransformationEstimationPointToPlane and TransformationEstimationColoredICP require pre-computed target normal vectors.");
    if (type != TransformationEstimationType::Unspecified) {
        cphb_cloud sc = source.view(), tc = target.view();
        cphb_icp_params p = make_params((int)type, max_correspondence_distance, criteria, estimation.det_thresh(), estimation.lambda_geometric());
        float T[16];
        utility::to_row_major(init, T);
        cphb_icp_result r;
        CorrespondenceSet corr(source.points_.size() ? source.points_.size() : 1);
        utility::check(cphb_registration_icp(&sc, &tc, T, &p, nullptr, &r, reinterpret_cast<int32_t *>(corr.data()), nullptr));
        return to_result(r, std::move(corr));
    }
    // generic loop (registration.cu:145-172) for user-subclassed estimators
    Eigen::Matrix4f transformation = init;
    geometry::PointCloud pcd = source;
    if (!init.isIdentity()) pcd.Transform(init);
    RegistrationResult result = EvaluateRegistration(pcd, target, max_correspondence_distance);
    result.transformation_ = transformation;
    for (int i = 0; i < criteria.max_iteration_; ++i) {
        Eigen::Matrix4f update = estimation.ComputeTransformation(pcd, target, result.correspondence_set_);
        transformation = update * transformation;
        pcd.Transform(update);
        const float bf = result.fitness_, br = result.inlier_rmse_;
        result = EvaluateRegistration(pcd, target, max_correspondence_distance);
        result.transformation_ = transformation;
        if (std::abs(bf - result.fitness_) < criteria.relative_fitness_ && std::abs(br - result.inlier_rmse_) < criteria.relative_rmse_) break;
    }
    return result;
}

/// InitializePointCloudForGeneralizedICP (generalized_icp.cu:37-61)
inline std::shared_ptr<geometry::PointCloud> InitializePointCloudForGeneralizedICP(const geometry::PointCloud &pcd, float epsilon) {
    auto out = std::make_shared<geometry::PointCloud>(pcd);
    if (out->HasCovariances()) return out;
    if (!out->HasNormals()) out->EstimateNormals(knn::KDTreeSearchParamKNN(20));
    out->covariances_.resize(out->points_.size());
    utility::check(cphb_covariances_from_normals(reinterpret_cast<const float *>(out->normals_.data()), out->points_.size(), epsilon,
                                                 reinterpret_cast<float *>(out->covariances_.data()), 1, nullptr));
    return out;
}
/// registration::RegistrationGeneralizedICP (generalized_icp.cu:185-198)
inline RegistrationResult RegistrationGeneralizedICP(const geometry::PointCloud &source, const geometry::PointCloud &target,
                                                     float max_correspondence_distance,
                                                     const Eigen::Matrix4f &init = Eigen::Matrix4f::Identity(),
                                                     const TransformationEstimationForGeneralizedICP &estimation = TransformationEstimationForGeneralizedICP(),
                                                     const ICPConvergenceCriteria &criteria = ICPConvergenceCriteria()) {
    return RegistrationICP(*InitializePointCloudForGeneralizedICP(source, estimation.epsilon_),
                           *InitializePointCloudForGeneralizedICP(target, estimation.epsilon_), max_correspondence_distance,
                           init, estimation, criteria);
}
/// registration::RegistrationColoredICP (colored_icp.cu:329-342)
inline RegistrationResult RegistrationColoredICP(const geometry::PointCloud &source, const geometry::PointCloud &target,
                                                 float max_distance, const Eigen::Matrix4f &init = Eigen::Matrix4f::Identity(),
                                                 const ICPConvergenceCriteria &criteria = ICPConvergenceCriteria(),
                                                 float lambda_geometric = 0.968, float det_thresh = 1.0e-6) {
    geometry::PointCloud target_c = target;  // InitializePointCloudForColoredICP (colored_icp.cu:120-148)
    target_c.color_gradient_.resize(target.points_.size());
    if (target.HasNormals() && target.HasColors())
        utility::check(cphb_color_gradient(reinterpret_cast<const float *>(target_c.points_.data()),
                                           reinterpret_cast<const float *>(target_c.normals_.data()),
                                           reinterpret_cast<const float *>(target_c.colors_.data()), target_c.points_.size(),
                                           max_distance * 2.0f, 30, reinterpret_cast<float *>(target_c.color_gradient_.data()), nullptr));
    else if (!target_c.color_gradient_.empty())
        utility::check(cphb_memset(target_c.color_gradient_.data(), 0, target_c.color_gradient_.size() * 12, nullptr));
    return RegistrationICP(source, target_c, max_distance, init, TransformationEstimationForColoredICP(lambda_geometric, det_thresh), criteria);
}
/// registration::Kabsch (kabsch.h:30-49)
inline Eigen::Matrix4f_u Kabsch(const utility::device_vector<Eigen::Vector3f> &model, const utility::device_vector<Eigen::Vector3f> &target,
                                const CorrespondenceSet &corres) {
    float T[16];
    utility::check(cphb_kabsch(reinterpret_cast<const float *>(model.data()), model.size(), reinterpret_cast<const float *>(target.data()),
                               reinterpret_cast<const int32_t *>(corres.data()), corres.size(), T, nullptr));
    return utility::from_row_major(T);
}
inline Eigen::Matrix4f_u Kabsch(const utility::device_vector<Eigen::Vector3f> &model, const utility::device_vector<Eigen::Vector3f> &target) {
    float T[16];
    utility::check(cphb_kabsch(reinterpret_cast<const float *>(model.data()), model.size(), reinterpret_cast<const float *>(target.data()),
                               nullptr, 0, T, nullptr));
    return utility::from_row_major(T);
}
/// registration::KabschWeighted (kabsch.h:46-49, kabsch.cu:138-201)
inline Eigen::Matrix4f_u KabschWeighted(const utility::device_vector<Eigen::Vector3f> &model,
                                        const utility::device_vector<Eigen::Vector3f> &target, const utility::device_vector<float> &weight) {
    float T[16];
    utility::check(cphb_kabsch_weighted(reinterpret_cast<const float *>(model.data()), reinterpret_cast<const float *>(target.data()),
                                        weight.data(), model.size(), T, nullptr));
    return utility::from_row_major(T);
}
/// registration::Feature<33> (feature.h): one row of 33 floats per point on the device
template <int Dim>
struct Feature {
    utility::device_vector<float> data_;
    size_t num_ = 0;
    void Resize(int n) { num_ = (size_t)n; data_.resize((size_t)n * Dim); }
    size_t Dimension() const { return Dim; }
    size_t Num() const { return num_; }
};
/// registration::ComputeFPFHFeature (feature.h, fpfh.cu:192-229)
inline std::shared_ptr<Feature<33>> ComputeFPFHFeature(const geometry::PointCloud &input,
                                                       const knn::KDTreeSearchParam &search_param = knn::KDTreeSearchParamKNN()) {
    auto feature = std::make_shared<Feature<33>>();
    feature->Resize((int)input.points_.size());
    if (!input.HasNormals()) {
        utility::LogError("[ComputeFPFHFeature] Failed because input point cloud has no normal.");
        return feature;
    }
    int knn = 0, max_nn = 0;
    float radius = 0.f;
    switch (search_param.GetSearchType()) {
        case knn::KDTreeSearchParam::SearchType::Knn: knn = ((const knn::KDTreeSearchParamKNN &)search_param).knn_; break;
        case knn::KDTreeSearchParam::SearchType::Radius:
            radius = ((const knn::KDTreeSearchParamRadius &)search_param).radius_;
            max_nn = ((const knn::KDTreeSearchParamRadius &)search_param).max_nn_;
            break;
        default: utility::LogError("Unsupport search param type."); return feature;
    }
    if (!input.points_.empty())
        utility::check(cphb_compute_fpfh_feature(reinterpret_cast<const float *>(input.points_.data()),
                                                 reinterpret_cast<const float *>(input.normals_.data()), input.points_.size(), knn, radius,
                                                 max_nn, feature->data_.data(), nullptr));
    return feature;
}

/// registration::FastGlobalRegistrationOption (fast_global_registration.h:43-104)
class FastGlobalRegistrationOption {
public:
    FastGlobalRegistrationOption(float division_factor = 1.4, bool use_absolute_scale = false, bool decrease_mu = true,
                                 float maximum_correspondence_distance = 0.025, int iteration_number = 64,
                                 float tuple_scale = 0.95, int maximum_tuple_count = 1000)
        : division_factor_(division_factor), use_absolute_scale_(use_absolute_scale), decrease_mu_(decrease_mu),
          maximum_correspondence_distance_(maximum_correspondence_distance), iteration_number_(iteration_number),
          tuple_scale_(tuple_scale), maximum_tuple_count_(maximum_tuple_count) {}
    float division_factor_;
    bool use_absolute_scale_;
    bool decrease_mu_;
    float maximum_correspondence_distance_;
    int iteration_number_;
    float tuple_scale_;
    int maximum_tuple_count_;
    cphb_fgr_option to_c() const {
        cphb_fgr_option o;
        o.division_factor = division_factor_;
        o.use_absolute_scale = use_absolute_scale_ ? 1 : 0;
        o.decrease_mu = decrease_mu_ ? 1 : 0;
        o.maximum_correspondence_distance = maximum_correspondence_distance_;
        o.iteration_number = iteration_number_;
        o.tuple_scale = tuple_scale_;
        o.maximum_tuple_count = maximum_tuple_count_;
        return o;
    }
};

/// registration::FastGlobalRegistration<Dim> (fast_global_registration.cu:391-431), Dim = 33 (FPFH) or 352 (SHOT)
template <int Dim>
inline RegistrationResult FastGlobalRegistration(const geometry::PointCloud &source, const geometry::PointCloud &target,
                                                 const Feature<Dim> &source_feature, const Feature<Dim> &target_feature,
                                                 const FastGlobalRegistrationOption &option = FastGlobalRegistrationOption()) {
    static_assert(Dim == 33 || Dim == 352, "FastGlobalRegistration supports Feature<33> and Feature<352>");
    if (source.points_.empty() || target.points_.empty() || source_feature.Num() == 0 || target_feature.Num() == 0) {
        utility::LogError("Invalid source or target pointcloud.");  // :400-404
        return RegistrationResult();
    }
    cphb_cloud sc = source.view(), tc = target.view();
    const cphb_fgr_option o = option.to_c();
    cphb_icp_result r;
    CorrespondenceSet corr(source.points_.size());
    utility::check(cphb_fast_global_registration(&sc, &tc, source_feature.data_.data(), source_feature.Num(),
                                                 target_feature.data_.data(), target_feature.Num(), Dim, &o, &r,
                                                 reinterpret_cast<int32_t *>(corr.data()), nullptr, nullptr));
    return to_result(r, std::move(corr));
}
}  // namespace registration

namespace knn {
/// knn::BruteForceNN<Dim>(ref, query, indices, distances) (bruteforce_nn.inl:101-135).  ref / query hold one row of
/// Dim floats per point (the layout of registration::Feature<Dim>::data_); exact, without a distance matrix.
template <int Dim>
inline void BruteForceNN(const utility::device_vector<float> &ref, const utility::device_vector<float> &query,
                         utility::device_vector<int> &indices, utility::device_vector<float> &distances) {
    static_assert(Dim == 33 || Dim == 352, "BruteForceNN supports Dim 33 and 352");
    const size_t nq = query.size() / Dim;
    indices.resize(nq);
    distances.resize(nq);
    if (nq == 0) return;
    utility::check(cphb_feature_nn(ref.data(), ref.size() / Dim, query.data(), nq, Dim, reinterpret_cast<int32_t *>(indices.data()),
                                   distances.data(), nullptr, nullptr, nullptr));
}
}  // namespace knn
}  // namespace cupoch
