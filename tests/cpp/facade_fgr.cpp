// FastGlobalRegistration and knn::BruteForceNN through the header-compatible facade, written the way the reference's
// examples call them: Feature<33> rows from ComputeFPFHFeature or from the caller, then
// registration::FastGlobalRegistration<33> with a FastGlobalRegistrationOption.
//   facade_fgr            : compile / link check only (no device needed to build)
//   facade_fgr DIR        : reads DIR/{src,tgt}.f32 ([n][3]) and DIR/{fs,ft}.f32 ([n][33]), writes DIR/T.f32 (4x4 row
//                           major), DIR/fit.f32 (fitness, inlier_rmse), DIR/corr.i32 and DIR/nn.i32 (BruteForceNN of
//                           ft against fs).  Exit code 0 = ran.
#include <cstdio>
#include <string>
#include <vector>

#include "cupoch/geometry/pointcloud.h"
#include "cupoch/knn/bruteforce_nn.h"
#include "cupoch/registration/fast_global_registration.h"
#include "cupoch/registration/registration.h"

using namespace cupoch;

template <class T>
static std::vector<T> read_all(const std::string &path) {
    std::vector<T> v;
    FILE *f = std::fopen(path.c_str(), "rb");
    if (!f) return v;
    std::fseek(f, 0, SEEK_END);
    const long bytes = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    v.resize((size_t)bytes / sizeof(T));
    if (std::fread(v.data(), sizeof(T), v.size(), f) != v.size()) v.clear();
    std::fclose(f);
    return v;
}
template <class T>
static void write_all(const std::string &path, const T *p, size_t n) {
    FILE *f = std::fopen(path.c_str(), "wb");
    if (!f) return;
    std::fwrite(p, sizeof(T), n, f);
    std::fclose(f);
}

int main(int argc, char **argv) {
    if (argc < 2) return 0;
    const std::string d = argv[1];
    auto s = read_all<float>(d + "/src.f32"), t = read_all<float>(d + "/tgt.f32");
    auto fs = read_all<float>(d + "/fs.f32"), ft = read_all<float>(d + "/ft.f32");
    std::vector<Eigen::Vector3f> sp(s.size() / 3), tp(t.size() / 3);
    for (size_t i = 0; i < sp.size(); ++i) sp[i] = Eigen::Vector3f(s[3 * i], s[3 * i + 1], s[3 * i + 2]);
    for (size_t i = 0; i < tp.size(); ++i) tp[i] = Eigen::Vector3f(t[3 * i], t[3 * i + 1], t[3 * i + 2]);
    geometry::PointCloud source, target;
    source.SetPoints(sp);
    target.SetPoints(tp);
    registration::Feature<33> f_s, f_t;
    f_s.Resize((int)sp.size());
    f_t.Resize((int)tp.size());
    f_s.data_ = fs;
    f_t.data_ = ft;
    registration::FastGlobalRegistrationOption option;
    option.maximum_correspondence_distance_ = 0.05f;
    option.iteration_number_ = 32;
    auto result = registration::FastGlobalRegistration<33>(source, target, f_s, f_t, option);
    float T[16];
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) T[4 * r + c] = result.transformation_(r, c);
    write_all(d + "/T.f32", T, 16);
    const float fit[2] = {result.fitness_, result.inlier_rmse_};
    write_all(d + "/fit.f32", fit, 2);
    auto corr = result.GetCorrespondenceSet();
    write_all(d + "/corr.i32", reinterpret_cast<const int *>(corr.data()), corr.size() * 2);
    utility::device_vector<int> idx;
    utility::device_vector<float> dist;
    knn::BruteForceNN<33>(f_s.data_, f_t.data_, idx, dist);
    auto h = idx.to_host();
    write_all(d + "/nn.i32", h.data(), h.size());
    return 0;
}
