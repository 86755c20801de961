// ct_icp_b200/odometry.hpp — header-only C++ facade with the API surface of ct_icp::Odometry
// (include/ct_icp/odometry.h:159-402 of the reference) over the C ABI in include/cticp.h.
//
// Same class, method, option and summary field names as the reference, so call sites such as
//   ct_icp::Odometry odometry(options);                                   command/odometry_runner.cpp:154
//   auto summary = odometry.RegisterFrame(frame, frame_id);               command/odometry_runner.cpp:194
//   trajectory.push_back(summary.frame.end_pose);                         command/odometry_runner.cpp:198
//   if (!summary.success) …                                               command/odometry_runner.cpp:276
// compile unchanged — including the slam::PointCloud overloads (any cloud type with size(), XYZConst<double>() and
// TimestampsProxy<double>(), the two views the reference reads, src/ct_icp/odometry.cpp:335-336), the AMotionModel*
// default arguments, RegisterCallback, Reset(options), Map() / MapConst().
// The reference's Eigen / SlamCore types are replaced by minimal PODs with the same member names
// (`pose.quat`, `pose.tr`, `dest_timestamp`, `RawPoint()`, `WorldPoint()`, `Timestamp()`): this header has no
// dependency besides cticp.h. INTEGRATION.md shows the variant that keeps the reference's own headers.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "cticp.h"

namespace slam {
typedef unsigned int frame_id_t;

struct Vec3d {   // stand-in for Eigen::Vector3d
    double v[3] = {0, 0, 0};
    double &operator[](int i) { return v[i]; }
    double operator[](int i) const { return v[i]; }
    double &x() { return v[0]; }
    double &y() { return v[1]; }
    double &z() { return v[2]; }
    double x() const { return v[0]; }
    double y() const { return v[1]; }
    double z() const { return v[2]; }
    double norm() const { return std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }
    Vec3d operator-(const Vec3d &o) const { return {{v[0] - o.v[0], v[1] - o.v[1], v[2] - o.v[2]}}; }
};
struct Quatd {   // stand-in for Eigen::Quaterniond (coefficients x, y, z, w)
    double c[4] = {0, 0, 0, 1};
    double x() const { return c[0]; }
    double y() const { return c[1]; }
    double z() const { return c[2]; }
    double w() const { return c[3]; }
    const double *coeffs() const { return c; }
};
struct SE3 {     // slam::TSE3<double>, include/SlamCore/types.h:100-139
    Quatd quat;
    Vec3d tr;
};
struct Pose {    // slam::TPose<double>, include/SlamCore/types.h:162-274
    SE3 pose;
    double ref_timestamp = 0, dest_timestamp = -1;
    frame_id_t ref_frame_id = 0, dest_frame_id = frame_id_t(-1);
    Quatd &QuatRef() { return pose.quat; }
    const Quatd &QuatConstRef() const { return pose.quat; }
    Vec3d &TrRef() { return pose.tr; }
    const Vec3d &TrConstRef() const { return pose.tr; }
};
struct Point3D {
    Vec3d point;
    double timestamp = -1;
};
struct WPoint3D {   // slam::WPoint3D, include/SlamCore/types.h:35-60
    Point3D raw_point;
    Vec3d world_point;
    frame_id_t index_frame = frame_id_t(-1);
    Vec3d &RawPoint() { return raw_point.point; }
    const Vec3d &RawPoint() const { return raw_point.point; }
    Vec3d &WorldPoint() { return world_point; }
    const Vec3d &WorldPoint() const { return world_point; }
    double &Timestamp() { return raw_point.timestamp; }
    const double &Timestamp() const { return raw_point.timestamp; }
};
static_assert(sizeof(WPoint3D) == sizeof(cticp_wpoint), "WPoint3D must keep the reference's 64-byte layout");
}  // namespace slam

namespace ct_icp {

enum CT_ICP_SOLVER { GN = CTICP_SOLVER_GN, CERES = CTICP_SOLVER_CERES, ROBUST = CTICP_SOLVER_ROBUST };
enum LEAST_SQUARES { STANDARD, CAUCHY, HUBER, TOLERANT, TRUNCATED };
enum MOTION_COMPENSATION { NONE = CTICP_MC_NONE, CONSTANT_VELOCITY, ITERATIVE, CONTINUOUS };
enum INITIALIZATION { INIT_NONE, INIT_CONSTANT_VELOCITY };

struct CticpFailure : std::runtime_error {
    int code;
    CticpFailure(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};
inline void cticp_check(int rc) {
    if (rc < 0) throw CticpFailure(rc, cticp_last_error());
}

// ct_icp::CTICPOptions (include/ct_icp/ct_icp.h:56-153): same field names; conversion is a memberwise copy
struct CTICPOptions : cticp_icp_options {
    CTICPOptions() { cticp_default_icp_options(this); }
};

// ct_icp::TrajectoryFrame, include/ct_icp/types.h:31-61
struct TrajectoryFrame {
    slam::Pose begin_pose, end_pose;
    const slam::Vec3d &BeginTr() const { return begin_pose.pose.tr; }
    const slam::Vec3d &EndTr() const { return end_pose.pose.tr; }
    const slam::Quatd &BeginQuat() const { return begin_pose.pose.quat; }
    const slam::Quatd &EndQuat() const { return end_pose.pose.quat; }
};

struct ICPSummary {   // include/ct_icp/ct_icp.h:155-169
    bool success = false;
    int num_residuals_used = 0, num_iters = 0;
    std::string error_log;
    double duration_total = 0, duration_init = 0, avg_duration_iter = 0, avg_duration_neighborhood = 0,
           avg_duration_solve = 0;
};

// ct_icp::OdometryOptions (include/ct_icp/odometry.h:32-157). The polymorphic map_options / neighborhood_strategy
// pointers of the reference are the embedded PODs `map_options` / `neighborhood_strategy`.
struct OdometryOptions : cticp_odometry_options {
    OdometryOptions() { cticp_default_odometry_options(this); }
    static OdometryOptions DefaultDrivingProfile() { OdometryOptions o; cticp_profile_default_driving(&o); return o; }
    static OdometryOptions RobustDrivingProfile() { OdometryOptions o; cticp_profile_robust_driving(&o); return o; }
    static OdometryOptions DefaultRobustOutdoorLowInertia() { OdometryOptions o; cticp_profile_robust_outdoor_low_inertia(&o); return o; }
};

namespace detail {
inline slam::Pose pose_from_c(const cticp_pose &c);
inline cticp_pose pose_to_c(const slam::Pose &p);
}

// ct_icp::AMotionModel / PreviousFrameMotionModel (include/ct_icp/motion_model.h:11-78): the state a caller-owned model
// carries into RegisterFrame. (AddConstraintsToCeresProblem has no meaning off Ceres: the engine adds the same four
// regularisers from `GetOptions()` and the previous frame.)
class AMotionModel {
public:
    virtual ~AMotionModel() = default;
    virtual void UpdateState(const TrajectoryFrame &optimized_frame, int frame_index) = 0;
    virtual void Reset() = 0;
    virtual bool ToPrior(cticp_motion_prior *out) const = 0;   // false: nothing to constrain with yet
};
class PreviousFrameMotionModel : public AMotionModel {
public:
    struct Options : cticp_motion_model_options {
        Options() {
            cticp_odometry_options o;
            cticp_default_odometry_options(&o);
            static_cast<cticp_motion_model_options &>(*this) = o.default_motion_model;
        }
    };
    PreviousFrameMotionModel() = default;
    explicit PreviousFrameMotionModel(const Options &options) : options_(options) {}
    void UpdateState(const TrajectoryFrame &optimized_frame, int) override {
        previous_frame_ = optimized_frame;
        has_frame_ = true;
    }
    void Reset() override { has_frame_ = false; }
    Options &GetOptions() { return options_; }
    const Options &GetOptions() const { return options_; }
    bool ToPrior(cticp_motion_prior *out) const override {
        if (!has_frame_) return false;
        out->options = options_;
        out->previous_frame.begin_pose = detail::pose_to_c(previous_frame_.begin_pose);
        out->previous_frame.end_pose = detail::pose_to_c(previous_frame_.end_pose);
        return true;
    }

private:
    Options options_;
    TrajectoryFrame previous_frame_;
    bool has_frame_ = false;
};

namespace detail {
inline slam::Pose pose_from_c(const cticp_pose &c) {
    slam::Pose p;
    std::memcpy(p.pose.quat.c, c.quat, sizeof(c.quat));
    std::memcpy(p.pose.tr.v, c.tr, sizeof(c.tr));
    p.ref_timestamp = c.ref_timestamp;
    p.dest_timestamp = c.dest_timestamp;
    p.ref_frame_id = c.ref_frame_id;
    p.dest_frame_id = c.dest_frame_id;
    return p;
}
inline cticp_pose pose_to_c(const slam::Pose &p) {
    cticp_pose c;
    std::memcpy(c.quat, p.pose.quat.c, sizeof(c.quat));
    std::memcpy(c.tr, p.pose.tr.v, sizeof(c.tr));
    c.ref_timestamp = p.ref_timestamp;
    c.dest_timestamp = p.dest_timestamp;
    c.ref_frame_id = p.ref_frame_id;
    c.dest_frame_id = p.dest_frame_id;
    return c;
}
inline TrajectoryFrame frame_from_c(const cticp_frame &c) { return {pose_from_c(c.begin_pose), pose_from_c(c.end_pose)}; }
inline cticp_frame frame_to_c(const TrajectoryFrame &f) { return {pose_to_c(f.begin_pose), pose_to_c(f.end_pose)}; }
}  // namespace detail

// ct_icp::ISlamMap view (include/ct_icp/map.h:14-83): the subset callers use through Odometry::GetMapPointer()
class MapView {
public:
    explicit MapView(cticp_map *m) : m_(m) {}
    size_t NumPoints() const { return (size_t) cticp_map_num_points(m_, 0); }                 // map.h:345
    std::vector<slam::Vec3d> MapAsPointCloud() const {                                         // map.h:350
        std::vector<slam::Vec3d> pts(NumPoints());
        if (!pts.empty()) cticp_map_export(m_, 0, &pts[0].v[0], nullptr, pts.size());
        return pts;
    }
    void RemoveElementsFarFromLocation(const slam::Vec3d &location, double distance) {         // map.h:305
        cticp_check(cticp_map_remove_far(m_, location.v, distance));
    }
    cticp_map *handle() const { return m_; }

private:
    cticp_map *m_;
};

class Odometry {
public:
    // The Output of a registration, including metrics (include/ct_icp/odometry.h:163-199)
    struct RegistrationSummary {
        TrajectoryFrame frame, initial_frame;
        int sample_size = 0, number_of_residuals = 0, robust_level = 0;
        double distance_correction = 0.0, relative_distance = 0.0, relative_orientation = 0.0, ego_orientation = 0.0;
        bool success = true, points_added = false;
        int number_of_attempts = 0;
        std::string error_message;
        std::vector<slam::WPoint3D> corrected_points, all_corrected_points, keypoints;
        ICPSummary icp_summary;
        std::map<std::string, double> logged_values;
    };

    // Which of the three point vectors RegisterFrame copies back from the device (the reference always fills all
    // three, odometry.cpp:462-486,597; a caller that only reads the poses can switch the copies off)
    struct CopyBack {
        bool corrected_points = true, all_corrected_points = true, keypoints = true;
    } copy_back;

    // An abstract Callback run at specified stages of the pipeline (include/ct_icp/odometry.h:206-224)
    struct OdometryCallback {
        enum EVENT { BEFORE_ITERATION, ITERATION_COMPLETED, FINISHED_REGISTRATION };
        virtual ~OdometryCallback() = default;
        virtual bool Run(const Odometry &odometry, const std::vector<slam::WPoint3D> &current_frame,
                         const std::vector<slam::WPoint3D> *keypoints = nullptr,
                         const RegistrationSummary *summary = nullptr) = 0;
    };

    explicit Odometry(const OdometryOptions &options, int device = 0) : options_(options) {
        cticp_check(cticp_odometry_create(&options, device, &h_));
        cticp_odometry_set_summary_points(h_, 7);   // the summary carries its three vectors by value: produce them eagerly
    }
    explicit Odometry(const OdometryOptions *options) : Odometry(*options) {}
    ~Odometry() { cticp_odometry_destroy(h_); }
    Odometry(const Odometry &) = delete;
    Odometry &operator=(const Odometry &) = delete;

    // Registers a new Frame to the Map (with custom motion model) (include/ct_icp/odometry.h:231-233). PointCloudT: the
    // reference's slam::PointCloud, or anything with its three accessors (tests/cpp/slam_pointcloud_stub.h)
    template <typename PointCloudT, typename = decltype(std::declval<const PointCloudT &>().template XYZConst<double>())>
    RegistrationSummary RegisterFrame(const PointCloudT &frame, slam::frame_id_t frame_id,
                                      AMotionModel *motion_model = nullptr) {
        return RegisterCloud(frame, frame_id, nullptr, motion_model);
    }
    // … with an initial estimate (:236-239)
    template <typename PointCloudT, typename = decltype(std::declval<const PointCloudT &>().template XYZConst<double>())>
    RegistrationSummary RegisterFrameWithEstimate(const PointCloudT &frame, const TrajectoryFrame &initial_estimate,
                                                  slam::frame_id_t frame_id, AMotionModel *motion_model = nullptr) {
        const cticp_frame est = detail::frame_to_c(initial_estimate);
        return RegisterCloud(frame, frame_id, &est, motion_model);
    }
    // Registers a new Frame to the Map (:242-243)
    RegistrationSummary RegisterFrame(const std::vector<slam::WPoint3D> &frame, AMotionModel *motion_model = nullptr) {
        return Register(frame, nullptr, frame.empty() ? 0 : frame.front().index_frame, motion_model);
    }
    // … with an initial estimate (:246-248)
    RegistrationSummary RegisterFrameWithEstimate(const std::vector<slam::WPoint3D> &frame,
                                                  const TrajectoryFrame &initial_estimate,
                                                  AMotionModel *motion_model = nullptr) {
        const cticp_frame est = detail::frame_to_c(initial_estimate);
        return Register(frame, &est, frame.empty() ? 0 : frame.front().index_frame, motion_model);
    }
    // strided arrays (what the PointCloud overload reads when its fields are already doubles)
    RegistrationSummary RegisterFrame(const double *xyz, size_t xyz_stride_bytes, const double *t,
                                      size_t t_stride_bytes, size_t n, slam::frame_id_t frame_id,
                                      AMotionModel *motion_model = nullptr) {
        return RegisterStrided(xyz, xyz_stride_bytes, t, t_stride_bytes, n, frame_id, nullptr, motion_model);
    }

    // Registers a Callback to the Odometry (:260; src/ct_icp/odometry.cpp:737-750)
    void RegisterCallback(OdometryCallback::EVENT event, OdometryCallback &callback) {
        callbacks_[event].push_back(&callback);
        cticp_check(cticp_odometry_set_callback(h_, &Odometry::Trampoline, this));
    }

    std::vector<TrajectoryFrame> Trajectory() const {   // :251
        const int64_t n = cticp_odometry_trajectory(h_, nullptr, 0);
        std::vector<cticp_frame> raw((size_t) n);
        cticp_odometry_trajectory(h_, raw.data(), raw.size());
        std::vector<TrajectoryFrame> out;
        out.reserve(raw.size());
        for (auto &f : raw) out.push_back(detail::frame_from_c(f));
        return out;
    }
    std::vector<slam::Vec3d> GetMapPointCloud() const { return MapView(cticp_odometry_map(h_)).MapAsPointCloud(); }   // :254
    size_t MapSize() const { return (size_t) cticp_odometry_map_size(h_); }                                           // :258
    MapView &Map() { map_view_ = MapView(cticp_odometry_map(h_)); return map_view_; }                                 // :263 REF_GETTER(Map, *map_)
    const MapView &MapConst() const { map_view_ = MapView(cticp_odometry_map(h_)); return map_view_; }
    void Reset() { cticp_check(cticp_odometry_reset(h_)); }                                                           // :266
    void Reset(const OdometryOptions &options) {                                                                      // :269
        cticp_check(cticp_odometry_reset_options(h_, &options));
        options_ = options;
        cticp_odometry_set_summary_points(h_, SummaryMask());
        if (!callbacks_.empty()) cticp_check(cticp_odometry_set_callback(h_, &Odometry::Trampoline, this));
    }
    std::shared_ptr<MapView> GetMapPointer() { return std::make_shared<MapView>(cticp_odometry_map(h_)); }            // :272
    // checkpoint / resume (new; cticp.h): a handle created with StateOptions(blob) that loads the blob continues the
    // saved run bit for bit
    std::vector<uint8_t> SaveState() const {
        const int64_t n = cticp_odometry_save_state(h_, nullptr, 0);
        cticp_check((int) std::min<int64_t>(n, 0));
        std::vector<uint8_t> blob((size_t) n);
        cticp_check((int) std::min<int64_t>(cticp_odometry_save_state(h_, blob.data(), blob.size()), 0));
        return blob;
    }
    void LoadState(const std::vector<uint8_t> &blob) { cticp_check(cticp_odometry_load_state(h_, blob.data(), blob.size())); }
    static OdometryOptions StateOptions(const std::vector<uint8_t> &blob) {
        OdometryOptions o;
        cticp_check(cticp_odometry_state_options(blob.data(), blob.size(), &o));
        return o;
    }
    const OdometryOptions &Options() const { return options_; }
    cticp_odometry *handle() const { return h_; }

private:
    int SummaryMask() const {
        return (copy_back.corrected_points ? 1 : 0) | (copy_back.all_corrected_points ? 2 : 0) | (copy_back.keypoints ? 4 : 0);
    }
    RegistrationSummary RegisterStrided(const double *xyz, size_t xyz_stride_bytes, const double *t, size_t t_stride_bytes,
                                        size_t n, slam::frame_id_t frame_id, const cticp_frame *estimate,
                                        AMotionModel *motion_model) {
        if (n == 0) throw std::invalid_argument("The registered frame cannot be empty");
        if (SummaryMask() != last_mask_) {
            cticp_odometry_set_summary_points(h_, SummaryMask());
            last_mask_ = SummaryMask();
        }
        cticp_motion_prior prior;
        const bool with_prior = motion_model && motion_model->ToPrior(&prior);
        cticp_summary s;
        cticp_check(cticp_odometry_register_frame_ex(h_, xyz, xyz_stride_bytes, t, t_stride_bytes, n, frame_id, estimate,
                                                     with_prior ? &prior : nullptr, &s));
        return MakeSummary(s);   // (like the reference, the caller's model is not updated here: the caller calls UpdateState)
    }
    RegistrationSummary Register(const std::vector<slam::WPoint3D> &frame, const cticp_frame *estimate,
                                 slam::frame_id_t frame_id, AMotionModel *motion_model) {
        if (frame.empty()) throw std::invalid_argument("The registered frame cannot be empty");
        return RegisterStrided(frame[0].raw_point.point.v, sizeof(slam::WPoint3D), &frame[0].raw_point.timestamp,
                               sizeof(slam::WPoint3D), frame.size(), frame_id, estimate, motion_model);
    }
    // the reference reads a PointCloud through two converting proxy views (any source scalar type); here they are
    // materialised as doubles once — the zero-copy route for sensor buffers is cticp_odometry_register_cloud
    template <typename PointCloudT>
    RegistrationSummary RegisterCloud(const PointCloudT &frame, slam::frame_id_t frame_id, const cticp_frame *estimate,
                                      AMotionModel *motion_model) {
        const size_t n = frame.size();
        const auto xyz = frame.template XYZConst<double>();
        const auto ts = frame.template TimestampsProxy<double>();
        scratch_.resize(4 * n);
        for (size_t i = 0; i < n; ++i) {
            const auto p = xyz[i];
            scratch_[4 * i] = p[0];
            scratch_[4 * i + 1] = p[1];
            scratch_[4 * i + 2] = p[2];
            scratch_[4 * i + 3] = ts[i];
        }
        return RegisterStrided(scratch_.data(), 32, scratch_.data() + 3, 32, n, frame_id, estimate, motion_model);
    }
    static int Trampoline(int event, void *user) {
        auto *self = static_cast<Odometry *>(user);
        auto it = self->callbacks_.find((typename OdometryCallback::EVENT) event);
        if (it == self->callbacks_.end() || it->second.empty()) return 1;
        std::vector<slam::WPoint3D> frame, keypoints;
        self->FetchAll(CTICP_POINTS_CORRECTED, frame);
        const bool with_kp = event != OdometryCallback::FINISHED_REGISTRATION;   // odometry.cpp:491,568,600
        if (with_kp) self->FetchAll(CTICP_POINTS_KEYPOINTS, keypoints);
        for (auto *cb : it->second)
            if (!cb->Run(*self, frame, with_kp ? &keypoints : nullptr, nullptr)) return 0;   // (:748 passes no summary)
        return 1;
    }
    void FetchAll(int which, std::vector<slam::WPoint3D> &dst) const {
        const int64_t n = cticp_odometry_get_points(h_, which, nullptr, 0);
        dst.resize(n > 0 ? (size_t) n : 0);
        if (n > 0) cticp_odometry_get_points(h_, which, reinterpret_cast<cticp_wpoint *>(dst.data()), dst.size());
    }
    void Fetch(int which, uint64_t count, std::vector<slam::WPoint3D> &dst) {
        dst.resize((size_t) count);
        if (count) cticp_odometry_get_points(h_, which, reinterpret_cast<cticp_wpoint *>(dst.data()), dst.size());
    }
    RegistrationSummary MakeSummary(const cticp_summary &s) {
        RegistrationSummary r;
        r.frame = detail::frame_from_c(s.frame);
        r.initial_frame = detail::frame_from_c(s.initial_frame);
        r.sample_size = s.sample_size;
        r.number_of_residuals = s.number_of_residuals;
        r.robust_level = s.robust_level;
        r.distance_correction = s.distance_correction;
        r.relative_distance = s.relative_distance;
        r.relative_orientation = s.relative_orientation;
        r.ego_orientation = s.ego_orientation;
        r.success = s.success != 0;
        r.points_added = s.points_added != 0;
        r.number_of_attempts = s.number_of_attempts;
        r.error_message = s.error_message;
        r.icp_summary.success = s.icp_summary.success != 0;
        r.icp_summary.num_residuals_used = s.icp_summary.num_residuals_used;
        r.icp_summary.num_iters = s.icp_summary.num_iters;
        r.icp_summary.error_log = s.error_message;
        r.icp_summary.duration_total = s.icp_summary.duration_total;
        r.icp_summary.duration_init = s.icp_summary.duration_init;
        r.icp_summary.avg_duration_iter = s.icp_summary.avg_duration_iter;
        r.icp_summary.avg_duration_neighborhood = s.icp_summary.avg_duration_neighborhood;
        r.icp_summary.avg_duration_solve = s.icp_summary.avg_duration_solve;
        // (all_corrected_points first: the engine sends it back first and in pieces, assembled while the rest is copying)
        if (copy_back.all_corrected_points) Fetch(CTICP_POINTS_ALL_CORRECTED, s.num_all_corrected_points, r.all_corrected_points);
        if (copy_back.keypoints) Fetch(CTICP_POINTS_KEYPOINTS, s.num_keypoints, r.keypoints);
        if (copy_back.corrected_points) Fetch(CTICP_POINTS_CORRECTED, s.num_corrected_points, r.corrected_points);
        // keys the ROS monitor consumes verbatim (ct_icp_odometry_node.cxx:279-287; odometry.cpp:495-513)
        r.logged_values["odometry_total"] = s.odometry_total;                              // :210
        r.logged_values["odometry_initialization"] = s.odometry_initialization;           // :211
        r.logged_values["odometry_total_duration(ms)"] = s.odometry_total;                // :496
        r.logged_values["odometry_initialization(ms)"] = s.odometry_initialization;       // :497
        r.logged_values["odometry_try_register"] = s.odometry_try_register;               // :428
        r.logged_values["odometry_duration_sampling"] = s.odometry_duration_sampling;     // :558
        r.logged_values["odometry_map_update(ms)"] = s.odometry_map_update;               // :498
        r.logged_values["odometry_transform(ms)"] = s.odometry_transform;                 // :499
        r.logged_values["odometry_num_keypoints"] = (double) s.num_keypoints;             // :495
        // LogSummary, :505-513
        r.logged_values["icp_duration_neighborhood"] = s.icp_summary.avg_duration_neighborhood * s.icp_summary.num_iters;
        r.logged_values["icp_duration_solve"] = s.icp_summary.avg_duration_solve * s.icp_summary.num_iters;
        r.logged_values["icp_total_duration"] = s.icp_summary.duration_total;
        r.logged_values["icp_num_iters"] = s.icp_summary.num_iters;
        return r;
    }
    cticp_odometry *h_ = nullptr;
    OdometryOptions options_;
    mutable MapView map_view_{nullptr};
    std::map<typename OdometryCallback::EVENT, std::vector<OdometryCallback *>> callbacks_;
    std::vector<double> scratch_;
    int last_mask_ = 7;
};

}  // namespace ct_icp
