// capi.cu — extern "C" entry points declared in include/cticp.h. No exceptions cross this boundary: every call
// returns a cticp_status and records its message for cticp_last_error().
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/cticp.h"
#include "engine.h"
#include "state_io.h"

using namespace cticp;

namespace {
thread_local std::string g_last_error;

int Fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
template <typename F>
int Guard(F &&f) {
    try {
        return f();
    } catch (const TimestampError &e) {
        return Fail(CTICP_ERR_TIMESTAMP, e.what());
    } catch (const UnsupportedError &e) {
        return Fail(CTICP_ERR_UNSUPPORTED, e.what());
    } catch (const CapacityError &e) {
        return Fail(CTICP_ERR_CAPACITY, e.what());
    } catch (const cticp::CallbackError &e) {
        return Fail(CTICP_ERR_CALLBACK, e.what());
    } catch (const CudaError &e) {
        return Fail(CTICP_ERR_CUDA, e.what());
    } catch (const std::invalid_argument &e) {
        return Fail(CTICP_ERR_INVALID_ARGUMENT, e.what());
    } catch (const std::runtime_error &e) {
        if (std::string(e.what()).rfind("NCCL", 0) == 0) return Fail(CTICP_ERR_NCCL, e.what());
        if (std::string(e.what()).rfind("NO_DEVICE", 0) == 0) return Fail(CTICP_ERR_NO_DEVICE, e.what());
        return Fail(CTICP_ERR_INTERNAL, e.what());
    } catch (const std::exception &e) {
        if (std::string(e.what()).rfind("NO_DEVICE", 0) == 0) return Fail(CTICP_ERR_NO_DEVICE, e.what());
        return Fail(CTICP_ERR_INTERNAL, e.what());
    }
}
#define CAPI_CUDA(expr)                                                                          \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) throw CudaError(std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

void RequireDevice(int device) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count)
        throw std::runtime_error("NO_DEVICE: no usable CUDA device (this engine has no CPU fallback)");
    CAPI_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CAPI_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) throw std::runtime_error("NO_DEVICE: this build targets sm_100a (Blackwell B200) only");
}
}  // namespace

struct cticp_map {
    DeviceMap *map = nullptr;
    IcpSolver *icp = nullptr;
    cudaStream_t stream = nullptr;
    int device = 0;
    bool owned = false;
};
struct cticp_odometry {
    Engine *engine = nullptr;
    cticp_map map_view;
};

extern "C" {

uint32_t cticp_abi_version(void) { return CTICP_ABI_VERSION; }
const char *cticp_last_error(void) { return g_last_error.c_str(); }

size_t cticp_abi_sizeof(const char *name) {
    const std::string s(name ? name : "");
    if (s == "cticp_icp_options") return sizeof(cticp_icp_options);
    if (s == "cticp_resolution_param") return sizeof(cticp_resolution_param);
    if (s == "cticp_map_options") return sizeof(cticp_map_options);
    if (s == "cticp_strategy_options") return sizeof(cticp_strategy_options);
    if (s == "cticp_motion_model_options") return sizeof(cticp_motion_model_options);
    if (s == "cticp_odometry_options") return sizeof(cticp_odometry_options);
    if (s == "cticp_pose") return sizeof(cticp_pose);
    if (s == "cticp_frame") return sizeof(cticp_frame);
    if (s == "cticp_wpoint") return sizeof(cticp_wpoint);
    if (s == "cticp_icp_summary") return sizeof(cticp_icp_summary);
    if (s == "cticp_summary") return sizeof(cticp_summary);
    if (s == "cticp_device_timing") return sizeof(cticp_device_timing);
    if (s == "cticp_adaptive_options") return sizeof(cticp_adaptive_options);
    return 0;
}

/* ---- defaults (include/ct_icp/ct_icp.h:60-152, map.h:115-125, odometry.h:37-157, motion_model.h:42-58) ------ */
void cticp_default_icp_options(cticp_icp_options *o) {
    memset(o, 0, sizeof(*o));
    o->num_iters_icp = 5;
    o->parametrization = CTICP_PARAM_CONTINUOUS_TIME;
    o->distance = CTICP_DIST_POINT_TO_PLANE;
    o->solver = CTICP_SOLVER_CERES;
    o->max_num_residuals = -1;
    o->min_num_residuals = 100;
    o->weighting_scheme = CTICP_WEIGHT_ALL;
    o->weight_alpha = 0.9;
    o->weight_neighborhood = 0.1;
    o->power_planarity = 2.0;
    o->max_number_neighbors = 20;
    o->min_number_neighbors = 20;
    o->threshold_voxel_occupancy = 1;
    o->num_closest_neighbors = 1;
    o->threshold_orientation_norm = 0.0001;
    o->threshold_translation_norm = 0.001;
    o->point_to_plane_with_distortion = 1;
    o->loss_function = CTICP_LOSS_CAUCHY;
    o->ls_max_num_iters = 1;
    o->ls_num_threads = 16;
    o->ls_sigma = 0.1;
    o->ls_tolerant_min_threshold = 0.05;
    o->max_dist_to_plane_ct_icp = 0.3;
    o->threshold_linearity = 0.8;
    o->threshold_planarity = 0.8;
    o->weight_point_to_point = 0.1;
    o->outlier_distance = 1.0;
    o->use_barycenter = 0;
    o->use_lines = 1;
    o->debug_print = 1;
}
void cticp_default_map_options(cticp_map_options *o) {
    memset(o, 0, sizeof(*o));
    o->num_resolutions = 3;
    o->resolutions[0].resolution = 0.2; o->resolutions[0].min_distance_between_points = 0.03; o->resolutions[0].max_num_points = 50;
    o->resolutions[1].resolution = 0.5; o->resolutions[1].min_distance_between_points = 0.1;  o->resolutions[1].max_num_points = 40;
    o->resolutions[2].resolution = 1.5; o->resolutions[2].min_distance_between_points = 0.15; o->resolutions[2].max_num_points = 40;
    o->select_valid_normals_direction = 1;
    o->max_frames_to_keep = 100;
    o->default_radius = 0.8;
}
void cticp_legacy_map_options(cticp_map_options *o, double size_voxel_map, int max_num_points_in_voxel,
                              double min_distance_points) {
    cticp_default_map_options(o);
    o->num_resolutions = 1;
    o->max_frames_to_keep = 1;
    o->resolutions[0].resolution = size_voxel_map;
    o->resolutions[0].max_num_points = max_num_points_in_voxel;
    o->resolutions[0].min_distance_between_points = min_distance_points;
}
void cticp_default_adaptive_options(cticp_adaptive_options *a) {   // include/ct_icp/algorithm/sampling.h:14-27
    memset(a, 0, sizeof(*a));
    a->num_points_per_voxel = 1;
    a->max_num_points = -1;
    a->num_bands = 6;
    const double d[6] = {0.5, 2.0, 4., 8., 16., 200.}, v[6] = {0.1, 0.2, 0.4, 0.8, 1.6, -1.};
    for (int i = 0; i < 6; ++i) {
        a->distance[i] = d[i];
        a->voxel_size[i] = v[i];
    }
}
void cticp_default_odometry_options(cticp_odometry_options *o) {
    memset(o, 0, sizeof(*o));
    cticp_default_adaptive_options(&o->adaptive_options);
    cticp_default_icp_options(&o->ct_icp_options);
    cticp_default_map_options(&o->map_options);
    o->neighborhood_strategy.type = 0;
    o->neighborhood_strategy.max_num_neighbors = 20;
    o->neighborhood_strategy.min_num_neighbors = 8;
    o->neighborhood_strategy.distance_max = 60.;   // DistanceBasedStrategy::Options, neighborhood_strategy.h:113-119
    o->neighborhood_strategy.radius_min = 0.1;
    o->neighborhood_strategy.radius_max = 2.0;
    o->neighborhood_strategy.exponent = 1.0;
    o->default_motion_model.model = CTICP_MM_CONSTANT_VELOCITY;
    o->default_motion_model.beta_location_consistency = 0.001;
    o->default_motion_model.beta_constant_velocity = 0.001;
    o->default_motion_model.beta_small_velocity = 0.0;
    o->default_motion_model.beta_orientation_consistency = 0.0;
    o->default_motion_model.threshold_orientation_deg = 15;
    o->default_motion_model.threshold_translation_diff = 0.3;
    o->default_motion_model.log_if_invalid = 1;
    o->motion_compensation = CTICP_MC_CONTINUOUS;
    o->initialization = CTICP_INIT_CONSTANT_VELOCITY;
    o->init_voxel_size = 0.2;
    o->init_sample_voxel_size = 1.0;
    o->init_num_frames = 20;
    o->sample_voxel_size = 1.5;
    o->max_num_keypoints = -1;
    o->sampling = CTICP_SAMPLING_GRID;
    o->voxel_size = 0.5;
    o->max_distance = 100.0;
    o->distance_error_threshold = 5.0;
    o->orientation_error_threshold = 30.;
    o->quit_on_error = 1;
    o->robust_minimal_level = 0;
    o->robust_registration = 0;
    o->robust_full_voxel_threshold = 0.7;
    o->robust_empty_voxel_threshold = 0.1;
    o->robust_neighborhood_min_dist = 0.10;
    o->robust_neighborhood_min_orientation = 0.1;
    o->robust_relative_trans_threshold = 1.0;
    o->robust_fail_early = 0;
    o->robust_num_attempts = 6;
    o->robust_num_attempts_when_rotation = 2;
    o->robust_max_voxel_neighborhood = 3;
    o->robust_threshold_ego_orientation = 3;
    o->robust_threshold_relative_orientation = 3;
    o->insertion_ego_rotation_threshold = 3;
    o->insertion_threshold_frames_skipped = 5;
    o->insertion_cum_distance_threshold = 0.8;
    o->insertion_cum_orientation_threshold = 5;
    o->always_insert = 0;
    o->do_no_insert = 0;
    o->debug_print = 1;
    o->with_default_motion_model = 1;
    o->shuffle_seed = 0x5DEECE66Dull;
    o->max_points_per_frame = 0;
}
void cticp_profile_default_driving(cticp_odometry_options *o) {
    cticp_default_odometry_options(o);
    o->ct_icp_options.solver = CTICP_SOLVER_CERES;
    o->ct_icp_options.ls_num_threads = 6;
    o->ct_icp_options.num_iters_icp = 5;
}
void cticp_profile_robust_driving(cticp_odometry_options *o) {
    cticp_default_odometry_options(o);
    o->voxel_size = 0.5;
    o->sample_voxel_size = 1.5;
    o->max_distance = 200.0;
    o->init_num_frames = 40;
    o->distance_error_threshold = 5.0;
    o->debug_print = 0;
    o->robust_registration = 1;
    o->robust_full_voxel_threshold = 0.5;
    o->robust_empty_voxel_threshold = 0.2;
    o->robust_num_attempts = 10;
    o->robust_max_voxel_neighborhood = 4;
    o->robust_threshold_relative_orientation = 5;
    o->robust_threshold_ego_orientation = 5;
    cticp_icp_options &c = o->ct_icp_options;
    c.debug_print = 0;
    c.max_number_neighbors = 20;
    c.min_number_neighbors = 20;
    c.num_iters_icp = 15;
    c.max_dist_to_plane_ct_icp = 0.5;
    c.threshold_orientation_norm = 0.01;
    c.num_closest_neighbors = 1;
    c.loss_function = CTICP_LOSS_CAUCHY;
    c.solver = CTICP_SOLVER_CERES;
    c.ls_max_num_iters = 20;
    c.ls_num_threads = 8;
    c.ls_sigma = 0.2;
    c.ls_tolerant_min_threshold = 0.05;
}
void cticp_profile_robust_outdoor_low_inertia(cticp_odometry_options *o) {
    cticp_default_odometry_options(o);
    o->voxel_size = 0.3;
    o->sample_voxel_size = 1.5;
    o->max_distance = 200.0;
    o->init_num_frames = 20;
    o->initialization = CTICP_INIT_NONE;
    o->debug_print = 0;
    o->robust_registration = 1;
    o->robust_full_voxel_threshold = 0.5;
    o->robust_empty_voxel_threshold = 0.1;
    o->robust_num_attempts = 3;
    o->robust_max_voxel_neighborhood = 4;
    o->robust_threshold_relative_orientation = 2;
    o->robust_threshold_ego_orientation = 2;
    o->default_motion_model.beta_constant_velocity = 0.0;
    o->default_motion_model.beta_location_consistency = 0.0;
    o->default_motion_model.beta_small_velocity = 0.001;
    o->default_motion_model.beta_orientation_consistency = 0.0;
    cticp_icp_options &c = o->ct_icp_options;
    c.num_iters_icp = 30;
    c.threshold_voxel_occupancy = 5;
    c.max_number_neighbors = 20;
    c.min_number_neighbors = 20;
    c.max_dist_to_plane_ct_icp = 0.5;
    c.threshold_orientation_norm = 0.01;
    c.num_closest_neighbors = 1;
    c.loss_function = CTICP_LOSS_CAUCHY;
    c.solver = CTICP_SOLVER_CERES;
    c.ls_max_num_iters = 10;
    c.ls_num_threads = 8;
    c.ls_sigma = 0.2;
    c.ls_tolerant_min_threshold = 0.05;
    c.weight_neighborhood = 0.2;
    c.weight_alpha = 0.8;
    c.weighting_scheme = CTICP_WEIGHT_ALL;
    c.max_num_residuals = 600;
    c.min_num_residuals = 200;
}

/* ---- Odometry ------------------------------------------------------------------------------------------------ */
int cticp_odometry_create(const cticp_odometry_options *options, int device, cticp_odometry **out) {
    return Guard([&] {
        if (!options || !out) throw std::invalid_argument("null argument");
        RequireDevice(device);
        auto *h = new cticp_odometry();
        try {
            h->engine = new Engine(*options, device);
        } catch (...) {
            delete h;
            throw;
        }
        h->map_view.map = &h->engine->Map();
        h->map_view.icp = &h->engine->Solver();
        h->map_view.stream = h->engine->Stream();
        h->map_view.device = device;
        h->map_view.owned = false;
        *out = h;
        return (int) CTICP_OK;
    });
}
void cticp_odometry_destroy(cticp_odometry *h) {
    if (!h) return;
    delete h->engine;
    delete h;
}
int cticp_odometry_register_frame(cticp_odometry *h, const double *xyz, size_t xyz_stride_bytes, const double *t,
                                  size_t t_stride_bytes, size_t n, uint32_t frame_id,
                                  const cticp_frame *initial_estimate, cticp_summary *out_summary) {
    return Guard([&] {
        if (!h) throw std::invalid_argument("null handle");
        cticp::ScanView v;
        v.xyz = xyz; v.xyz_stride = xyz_stride_bytes; v.t = t; v.t_stride = t_stride_bytes; v.n = n;
        h->engine->RegisterFrame(v, frame_id, initial_estimate, out_summary);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_register_frame_ex(cticp_odometry *h, const double *xyz, size_t xyz_stride_bytes, const double *t,
                                     size_t t_stride_bytes, size_t n, uint32_t frame_id,
                                     const cticp_frame *initial_estimate, const cticp_motion_prior *motion_model,
                                     cticp_summary *out_summary) {
    return Guard([&] {
        if (!h) throw std::invalid_argument("null handle");
        cticp::ScanView v;
        v.xyz = xyz; v.xyz_stride = xyz_stride_bytes; v.t = t; v.t_stride = t_stride_bytes; v.n = n;
        h->engine->RegisterFrame(v, frame_id, initial_estimate, out_summary, motion_model);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_set_callback(cticp_odometry *h, cticp_event_fn fn, void *user) {
    return Guard([&] {
        if (!h) throw std::invalid_argument("null handle");
        h->engine->SetCallback(fn, user);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_reset_options(cticp_odometry *h, const cticp_odometry_options *options) {
    return Guard([&] {
        if (!h || !options) throw std::invalid_argument("null argument");
        const int device = h->engine->Device();
        Engine *fresh = new Engine(*options, device);   // throws before the old engine is touched
        delete h->engine;
        h->engine = fresh;
        h->map_view.map = &h->engine->Map();
        h->map_view.icp = &h->engine->Solver();
        h->map_view.stream = h->engine->Stream();
        return (int) CTICP_OK;
    });
}
static cticp::ScanView ViewOfCloud(const cticp_cloud_view *c) {
    if (!c || !c->data) throw std::invalid_argument("The registered frame cannot be empty");
    const size_t xs = c->xyz_dtype == CTICP_DTYPE_FLOAT32 ? 4 : 8;
    static const size_t kSize[9] = {0, 1, 1, 2, 2, 4, 4, 4, 8};
    if (c->t_dtype < 1 || c->t_dtype > 8) throw std::invalid_argument("unknown timestamp dtype");
    if ((size_t) c->xyz_offset + 3 * xs > c->point_step || (size_t) c->t_offset + kSize[c->t_dtype] > c->point_step)
        throw std::invalid_argument("cloud view: a field lies outside the record (point_step)");
    cticp::ScanView v;
    v.xyz = static_cast<const char *>(c->data) + c->xyz_offset;
    v.xyz_stride = c->point_step;
    v.xyz_dtype = c->xyz_dtype;
    v.t = static_cast<const char *>(c->data) + c->t_offset;
    v.t_stride = c->point_step;
    v.t_dtype = c->t_dtype;
    v.n = (size_t) c->num_points;
    return v;
}
int cticp_odometry_register_cloud(cticp_odometry *h, const cticp_cloud_view *cloud, uint32_t frame_id,
                                  const cticp_frame *initial_estimate, cticp_summary *out_summary) {
    return Guard([&] {
        if (!h) throw std::invalid_argument("null handle");
        h->engine->RegisterFrame(ViewOfCloud(cloud), frame_id, initial_estimate, out_summary);
        return (int) CTICP_OK;
    });
}
int64_t cticp_odometry_stage_cloud(cticp_odometry *h, const cticp_cloud_view *cloud) {
    int64_t slot = -1;
    int rc = Guard([&] {
        slot = h->engine->StageFrame(ViewOfCloud(cloud));
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : slot;
}
int64_t cticp_odometry_write_points(cticp_odometry *h, int which, const cticp_cloud_sink *sink) {
    int64_t count = 0;
    int rc = Guard([&] {
        if (!sink) throw std::invalid_argument("null sink");
        count = h->engine->WritePoints(which, *sink);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : count;
}
int64_t cticp_odometry_get_points(cticp_odometry *h, int which, cticp_wpoint *dst, size_t cap) {
    int64_t count = 0;
    int rc = Guard([&] {
        count = h->engine->GetPoints(which, dst, cap);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : count;
}
int cticp_odometry_set_summary_points(cticp_odometry *h, int mask) {
    return Guard([&] {
        h->engine->SetSummaryPoints(mask);
        return (int) CTICP_OK;
    });
}
int64_t cticp_odometry_trajectory(cticp_odometry *h, cticp_frame *dst, size_t cap) {
    const auto &tr = h->engine->Trajectory();
    const size_t m = std::min(cap, tr.size());
    for (size_t i = 0; i < m && dst; ++i) dst[i] = FrameToC(tr[i]);
    return (int64_t) tr.size();
}
int64_t cticp_odometry_map_size(cticp_odometry *h) {
    int64_t v = 0;
    int rc = Guard([&] {
        v = h->engine->MapSize();
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : v;
}
int64_t cticp_odometry_map_points(cticp_odometry *h, double *dst_xyz, size_t cap_points) {
    return cticp_map_export(&h->map_view, 0, dst_xyz, nullptr, cap_points);
}
int cticp_odometry_reset(cticp_odometry *h) {
    return Guard([&] {
        h->engine->Reset();
        return (int) CTICP_OK;
    });
}
cticp_map *cticp_odometry_map(cticp_odometry *h) { return h ? &h->map_view : nullptr; }
int cticp_odometry_last_timing(cticp_odometry *h, cticp_device_timing *out) {
    return Guard([&] {
        *out = h->engine->LastTiming();
        return (int) CTICP_OK;
    });
}
int64_t cticp_odometry_stage_frame(cticp_odometry *h, const double *xyz, size_t xyz_stride_bytes, const double *t,
                                   size_t t_stride_bytes, size_t n) {
    int64_t slot = -1;
    int rc = Guard([&] {
        cticp::ScanView v;
        v.xyz = xyz; v.xyz_stride = xyz_stride_bytes; v.t = t; v.t_stride = t_stride_bytes; v.n = n;
        slot = h->engine->StageFrame(v);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : slot;
}
int cticp_odometry_register_staged(cticp_odometry *h, int64_t slot, uint32_t frame_id, cticp_summary *out_summary) {
    return Guard([&] {
        h->engine->RegisterStaged(slot, frame_id, out_summary);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_clear_staged(cticp_odometry *h) {
    return Guard([&] {
        h->engine->ClearStaged();
        return (int) CTICP_OK;
    });
}
int cticp_odometry_timer_start(cticp_odometry *h) {
    return Guard([&] {
        h->engine->TimerStart();
        return (int) CTICP_OK;
    });
}
int cticp_odometry_timer_stop(cticp_odometry *h, double *elapsed_ms) {
    return Guard([&] {
        *elapsed_ms = h->engine->TimerStop();
        return (int) CTICP_OK;
    });
}
int cticp_odometry_flush_l2(cticp_odometry *h, size_t bytes) {
    return Guard([&] {
        h->engine->FlushL2(bytes);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_set_gather_timing(cticp_odometry *h, int on) {
    h->engine->SetTimeGather(on != 0);
    return CTICP_OK;
}
int cticp_odometry_enable_sharding(cticp_odometry *h, const void *unique_id_128_bytes, int rank, int world) {
    return Guard([&] {
        h->engine->EnableSharding(unique_id_128_bytes, rank, world);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_sharding_mode(cticp_odometry *h) { return h->engine->ShardingMode(); }

/* ---- checkpoint / resume (state_io.h) ------------------------------------------------------------------------- */
int64_t cticp_odometry_save_state(cticp_odometry *h, void *dst, size_t cap) {
    int64_t size = 0;
    int rc = Guard([&] {
        if (!h) throw std::invalid_argument("null handle");
        size = h->engine->SaveState(static_cast<uint8_t *>(dst), cap);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : size;
}
int cticp_odometry_load_state(cticp_odometry *h, const void *src, size_t size) {
    return Guard([&] {
        if (!h) throw std::invalid_argument("null handle");
        h->engine->LoadState(static_cast<const uint8_t *>(src), size);
        return (int) CTICP_OK;
    });
}
int cticp_odometry_state_options(const void *src, size_t size, cticp_odometry_options *out) {
    return Guard([&] {
        if (!out) throw std::invalid_argument("null argument");
        *out = OdoParse(static_cast<const uint8_t *>(src), size, false).options;
        return (int) CTICP_OK;
    });
}

/* ---- Map ----------------------------------------------------------------------------------------------------- */
int cticp_map_create(const cticp_map_options *options, int device, cticp_map **out) {
    return Guard([&] {
        if (!options || !out) throw std::invalid_argument("null argument");
        RequireDevice(device);
        auto *m = new cticp_map();
        m->device = device;
        m->owned = true;
        CAPI_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
        m->map = new DeviceMap(*options, m->stream, options->select_valid_normals_direction != 0);
        m->icp = new IcpSolver(m->stream);
        CAPI_CUDA(cudaStreamSynchronize(m->stream));
        *out = m;
        return (int) CTICP_OK;
    });
}
void cticp_map_destroy(cticp_map *m) {
    if (!m || !m->owned) return;
    cudaSetDevice(m->device);
    cudaStreamSynchronize(m->stream);
    delete m->icp;
    delete m->map;
    cudaStreamDestroy(m->stream);
    delete m;
}
int cticp_map_insert(cticp_map *m, const double *xyz, size_t stride_bytes, size_t n) {
    return cticp_map_insert_from(m, xyz, stride_bytes, n, nullptr);
}
int cticp_map_insert_from(cticp_map *m, const double *xyz, size_t stride_bytes, size_t n, const double origin[3]) {
    return Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        m->map->InsertHost(xyz, stride_bytes, n, origin ? V3{origin[0], origin[1], origin[2]} : V3{0, 0, 0});
        m->map->SyncCounters();
        m->map->MaintainTables();
        return (int) CTICP_OK;
    });
}
int cticp_map_remove_far(cticp_map *m, const double location[3], double distance) {
    return Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        m->map->RemoveFar(V3{location[0], location[1], location[2]}, distance);
        m->map->SyncCounters();
        m->map->MaintainTables();
        return (int) CTICP_OK;
    });
}
int64_t cticp_map_num_points(cticp_map *m, int map_idx) {
    int64_t v = 0;
    int rc = Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        if (map_idx < 0 || map_idx >= m->map->NumLevels()) throw std::invalid_argument("map_idx");
        v = (int64_t) m->map->SyncCounters()[map_idx].num_points;
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : v;
}
int64_t cticp_map_num_voxels(cticp_map *m, int map_idx) {
    int64_t v = 0;
    int rc = Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        if (map_idx < 0 || map_idx >= m->map->NumLevels()) throw std::invalid_argument("map_idx");
        v = (int64_t) m->map->SyncCounters()[map_idx].num_voxels;
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : v;
}
int64_t cticp_map_export(cticp_map *m, int map_idx, double *dst_xyz, int32_t *dst_voxel, size_t cap_points) {
    int64_t v = 0;
    int rc = Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        if (map_idx < 0 || map_idx >= m->map->NumLevels()) throw std::invalid_argument("map_idx");
        std::vector<double> xyz;
        std::vector<int> vox;
        const size_t n = m->map->Export(map_idx, xyz, vox);
        const size_t k = std::min(cap_points, n);
        if (dst_xyz) memcpy(dst_xyz, xyz.data(), sizeof(double) * 3 * k);
        if (dst_voxel) memcpy(dst_voxel, vox.data(), sizeof(int32_t) * 3 * k);
        v = (int64_t) n;
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : v;
}
int cticp_map_compute_neighborhoods(cticp_map *m, const double *queries_xyz, size_t n, int max_num_neighbors,
                                    double *out_points, int32_t *out_counts) {
    return Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        if (n == 0) return (int) CTICP_OK;
        double *d_q, *d_out;
        int *d_cnt;
        CAPI_CUDA(cudaMalloc(&d_q, sizeof(double) * 3 * n));
        CAPI_CUDA(cudaMalloc(&d_out, sizeof(double) * 3 * n * max_num_neighbors));
        CAPI_CUDA(cudaMalloc(&d_cnt, sizeof(int) * n));
        CAPI_CUDA(cudaMemcpyAsync(d_q, queries_xyz, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, m->stream));
        CAPI_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * 3 * n * max_num_neighbors, m->stream));
        m->icp->Neighborhoods(*m->map, d_q, n, max_num_neighbors, d_out, d_cnt);
        CAPI_CUDA(cudaMemcpyAsync(out_points, d_out, sizeof(double) * 3 * n * max_num_neighbors, cudaMemcpyDeviceToHost, m->stream));
        CAPI_CUDA(cudaMemcpyAsync(out_counts, d_cnt, sizeof(int) * n, cudaMemcpyDeviceToHost, m->stream));
        CAPI_CUDA(cudaStreamSynchronize(m->stream));
        cudaFree(d_q); cudaFree(d_out); cudaFree(d_cnt);
        return (int) CTICP_OK;
    });
}
int cticp_map_radius_search(cticp_map *m, const double *queries_xyz, const double *radiuses, size_t n,
                            int max_num_neighbors, const double *sensor_location, double *out_points,
                            int32_t *out_counts) {
    return Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        if (n == 0) return (int) CTICP_OK;
        if (!queries_xyz || !radiuses || !out_points || !out_counts) throw std::invalid_argument("null argument");
        double *d_q, *d_r, *d_out;
        int *d_cnt;
        CAPI_CUDA(cudaMalloc(&d_q, sizeof(double) * 3 * n));
        CAPI_CUDA(cudaMalloc(&d_r, sizeof(double) * n));
        CAPI_CUDA(cudaMalloc(&d_out, sizeof(double) * 3 * n * max_num_neighbors));
        CAPI_CUDA(cudaMalloc(&d_cnt, sizeof(int) * n));
        CAPI_CUDA(cudaMemcpyAsync(d_q, queries_xyz, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, m->stream));
        CAPI_CUDA(cudaMemcpyAsync(d_r, radiuses, sizeof(double) * n, cudaMemcpyHostToDevice, m->stream));
        CAPI_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * 3 * n * max_num_neighbors, m->stream));
        m->icp->RadiusSearch(*m->map, d_q, d_r, n, max_num_neighbors, sensor_location, d_out, d_cnt);
        CAPI_CUDA(cudaMemcpyAsync(out_points, d_out, sizeof(double) * 3 * n * max_num_neighbors, cudaMemcpyDeviceToHost, m->stream));
        CAPI_CUDA(cudaMemcpyAsync(out_counts, d_cnt, sizeof(int) * n, cudaMemcpyDeviceToHost, m->stream));
        CAPI_CUDA(cudaStreamSynchronize(m->stream));
        cudaFree(d_q); cudaFree(d_r); cudaFree(d_out); cudaFree(d_cnt);
        return (int) CTICP_OK;
    });
}
int64_t cticp_map_save(cticp_map *m, void *dst, size_t cap) {
    int64_t size = 0;
    int rc = Guard([&] {
        if (!m) throw std::invalid_argument("null handle");
        CAPI_CUDA(cudaSetDevice(m->device));
        size = (int64_t) m->map->Save(static_cast<uint8_t *>(dst), cap);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : size;
}
int cticp_map_load(cticp_map *m, const void *src, size_t size) {
    return Guard([&] {
        if (!m) throw std::invalid_argument("null handle");
        // the odometry's own map changes together with the trajectory and the policy state that refer to it
        if (!m->owned) throw UnsupportedError("map load: this map belongs to an odometry; load the odometry's state instead");
        CAPI_CUDA(cudaSetDevice(m->device));
        m->map->Load(static_cast<const uint8_t *>(src), size);
        return (int) CTICP_OK;
    });
}
int cticp_map_clear(cticp_map *m) {
    return Guard([&] {
        CAPI_CUDA(cudaSetDevice(m->device));
        m->map->Clear();
        m->map->SyncCounters();
        return (int) CTICP_OK;
    });
}

/* ---- Registration -------------------------------------------------------------------------------------------- */
namespace {
// TPose::GetAlphaTimestamp (types.h:192-219)
double AlphaOf(double t, double bts, double ets) {
    const double mn = std::min(bts, ets), mx = std::max(bts, ets);
    if (mn > t || mx < t) return 0.0;
    if (mn == mx) return 1.0;
    return (t - mn) / (mx - mn);
}
struct DeviceKeypoints {
    float4 *d_kp = nullptr;
    float4 *d_lo = nullptr;   // residual plane (se3.cuh load_raw); has_lo: some coordinate is not float32-representable
    bool has_lo = false;
    int *d_n = nullptr;
    IcpState *d_state = nullptr;
    const float4 *lo() const { return has_lo ? d_lo : nullptr; }
    ~DeviceKeypoints() {
        cudaFree(d_kp);
        cudaFree(d_lo);
        cudaFree(d_n);
        cudaFree(d_state);
    }
};
void UploadRegistrationInputs(cticp_map *m, const cticp_wpoint *keypoints, size_t n, const cticp_frame *frame,
                              const cticp_frame *previous_frame, const cticp_motion_model_options *mo,
                              DeviceKeypoints &D, IcpState &S) {
    const double bts = frame->begin_pose.dest_timestamp, ets = frame->end_pose.dest_timestamp;
    std::vector<float4> kp(n), lo(n);
    for (size_t i = 0; i < n; ++i) {
        const double t = keypoints[i].timestamp;
        if (!(bts <= t && t <= ets)) throw TimestampError("The timestamp cannot be interpolated between the two poses");
        const double v[4] = {keypoints[i].raw[0], keypoints[i].raw[1], keypoints[i].raw[2], AlphaOf(t, bts, ets)};
        kp[i] = make_float4((float) v[0], (float) v[1], (float) v[2], (float) v[3]);
        lo[i] = make_float4((float) (v[0] - (double) kp[i].x), (float) (v[1] - (double) kp[i].y),
                            (float) (v[2] - (double) kp[i].z), (float) (v[3] - (double) kp[i].w));
        if (lo[i].x != 0.f || lo[i].y != 0.f || lo[i].z != 0.f || lo[i].w != 0.f) D.has_lo = true;
    }
    CAPI_CUDA(cudaMalloc(&D.d_kp, sizeof(float4) * std::max<size_t>(n, 1)));
    CAPI_CUDA(cudaMalloc(&D.d_lo, sizeof(float4) * std::max<size_t>(n, 1)));
    CAPI_CUDA(cudaMemcpyAsync(D.d_lo, lo.data(), sizeof(float4) * n, cudaMemcpyHostToDevice, m->stream));
    CAPI_CUDA(cudaMalloc(&D.d_n, sizeof(int)));
    CAPI_CUDA(cudaMalloc(&D.d_state, sizeof(IcpState)));
    const int ni = (int) n;
    memset(&S, 0, sizeof(S));
    const Q4 qb = qnormalized(Q4{frame->begin_pose.quat[0], frame->begin_pose.quat[1], frame->begin_pose.quat[2], frame->begin_pose.quat[3]});
    const Q4 qe = qnormalized(Q4{frame->end_pose.quat[0], frame->end_pose.quat[1], frame->end_pose.quat[2], frame->end_pose.quat[3]});
    S.qb[0] = qb.x; S.qb[1] = qb.y; S.qb[2] = qb.z; S.qb[3] = qb.w;
    S.qe[0] = qe.x; S.qe[1] = qe.y; S.qe[2] = qe.z; S.qe[3] = qe.w;
    for (int d = 0; d < 3; ++d) {
        S.tb[d] = frame->begin_pose.tr[d];
        S.te[d] = frame->end_pose.tr[d];
    }
    if (previous_frame && mo) {
        S.has_motion_model = 1;
        S.beta_location = mo->beta_location_consistency;
        S.beta_cv = mo->beta_constant_velocity;
        S.beta_small = mo->beta_small_velocity;
        S.beta_orientation = mo->beta_orientation_consistency;
        for (int d = 0; d < 3; ++d) {
            S.prev_tb[d] = previous_frame->begin_pose.tr[d];
            S.prev_te[d] = previous_frame->end_pose.tr[d];
        }
        for (int d = 0; d < 4; ++d) S.prev_qe[d] = previous_frame->end_pose.quat[d];
    }
    icp_state_refresh_slerp(S);
    CAPI_CUDA(cudaMemcpyAsync(D.d_kp, kp.data(), sizeof(float4) * n, cudaMemcpyHostToDevice, m->stream));
    CAPI_CUDA(cudaMemcpyAsync(D.d_n, &ni, sizeof(int), cudaMemcpyHostToDevice, m->stream));
    CAPI_CUDA(cudaMemcpyAsync(D.d_state, &S, sizeof(IcpState), cudaMemcpyHostToDevice, m->stream));
    CAPI_CUDA(cudaStreamSynchronize(m->stream));
}
}  // namespace

int cticp_icp_register(cticp_map *m, const cticp_icp_options *options, const cticp_strategy_options *strategy,
                       cticp_wpoint *keypoints, size_t n, cticp_frame *frame, const cticp_frame *previous_frame,
                       const cticp_motion_model_options *motion_options, cticp_icp_summary *out_summary) {
    return Guard([&] {
        if (!m || !options || !keypoints || !frame) throw std::invalid_argument("null argument");
        CAPI_CUDA(cudaSetDevice(m->device));
        DeviceKeypoints D;
        IcpState S;
        UploadRegistrationInputs(m, keypoints, n, frame, previous_frame, motion_options, D, S);
        cticp_strategy_options st{0, 20, 8, 0, 60., 0.1, 2.0, 1.0};
        if (strategy) st = *strategy;
        m->icp->set_keypoints_lo(D.lo());
        switch (options->solver) {
            case CTICP_SOLVER_GN:
                m->icp->EnqueueGaussNewton(*m->map, *options, D.d_kp, D.d_n, n, options->num_iters_icp, D.d_state);
                break;
            case CTICP_SOLVER_CERES:
            case CTICP_SOLVER_ROBUST:
                m->icp->EnqueueCeres(*m->map, *options, st, D.d_kp, D.d_n, n, n, D.d_state);
                break;
            default:
                throw UnsupportedError("Unsupported Solver Type");
        }
        CAPI_CUDA(cudaMemcpyAsync(&S, D.d_state, sizeof(IcpState), cudaMemcpyDeviceToHost, m->stream));
        CAPI_CUDA(cudaStreamSynchronize(m->stream));
        for (int d = 0; d < 4; ++d) {
            frame->begin_pose.quat[d] = S.qb[d];
            frame->end_pose.quat[d] = S.qe[d];
        }
        for (int d = 0; d < 3; ++d) {
            frame->begin_pose.tr[d] = S.tb[d];
            frame->end_pose.tr[d] = S.te[d];
        }
        // world_kpts[i] ← InterpolatePose(begin, end, t_i) * raw_i with the final pose pair (ct_icp.cpp:964-966, :688)
        const Q4 qb{S.qb[0], S.qb[1], S.qb[2], S.qb[3]}, qe{S.qe[0], S.qe[1], S.qe[2], S.qe[3]};
        const V3 tb{S.tb[0], S.tb[1], S.tb[2]}, te{S.te[0], S.te[1], S.te[2]};
        const double bts = frame->begin_pose.dest_timestamp, ets = frame->end_pose.dest_timestamp;
        for (size_t i = 0; i < n; ++i) {
            const V3 w = ct_transform(qb, tb, qe, te, AlphaOf(keypoints[i].timestamp, bts, ets),
                                      V3{keypoints[i].raw[0], keypoints[i].raw[1], keypoints[i].raw[2]});
            keypoints[i].world[0] = w.x; keypoints[i].world[1] = w.y; keypoints[i].world[2] = w.z;
        }
        if (out_summary) {
            memset(out_summary, 0, sizeof(*out_summary));
            out_summary->success = !S.failed;
            out_summary->num_residuals_used = S.n_used;
            out_summary->num_iters = S.iter;
        }
        if (S.failed == 2) throw std::runtime_error("Error During Optimization");
        if (S.failed) g_last_error = "[CT_ICP]Error : not enough keypoints selected in ct-icp !";
        return (int) CTICP_OK;
    });
}

int cticp_icp_gn_normal_equations(cticp_map *m, const cticp_icp_options *options, const cticp_wpoint *keypoints,
                                  size_t n, const cticp_frame *frame, const cticp_frame *previous_frame,
                                  const cticp_motion_model_options *motion_options, double *out_A144, double *out_b12,
                                  int32_t *out_num_used) {
    return Guard([&] {
        if (!m || !options || !keypoints || !frame) throw std::invalid_argument("null argument");
        CAPI_CUDA(cudaSetDevice(m->device));
        DeviceKeypoints D;
        IcpState S;
        UploadRegistrationInputs(m, keypoints, n, frame, previous_frame, motion_options, D, S);
        int n_used = 0;
        m->icp->set_keypoints_lo(D.lo());
        m->icp->NormalEquations(*m->map, *options, D.d_kp, D.d_n, n, D.d_state, out_A144, out_b12, &n_used);
        *out_num_used = n_used;
        return (int) CTICP_OK;
    });
}

/* ---- Sampling / order contract ------------------------------------------------------------------------------- */
int64_t cticp_grid_sample_indices(int device, const double *xyz, size_t stride_bytes, size_t n, double voxel_size,
                                  uint32_t *out_indices, size_t cap) {
    int64_t total = 0;
    int rc = Guard([&] {
        RequireDevice(device);
        if (n == 0) return (int) CTICP_OK;
        cudaStream_t stream;
        CAPI_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        {
            FramePipeline pipe(n, stream);
            float4 *stage = pipe.Staging(), *stage_lo = pipe.StagingLo();
            for (size_t i = 0; i < n; ++i) {
                const double *p = reinterpret_cast<const double *>(reinterpret_cast<const char *>(xyz) + stride_bytes * i);
                stage[i] = make_float4((float) p[0], (float) p[1], (float) p[2], 0.f);
                stage_lo[i] = make_float4((float) (p[0] - (double) stage[i].x), (float) (p[1] - (double) stage[i].y),
                                          (float) (p[2] - (double) stage[i].z), 0.f);
            }
            pipe.Upload(n);
            pipe.UploadLo(n);
            pipe.GridSelect(pipe.d_raw(), pipe.d_raw_lo(), nullptr, pipe.d_count_n(), n, voxel_size, 0, 0, 0, 0, 0, 0, 0.f,
                            pipe.d_frame_mut(), pipe.d_frame_lo_mut(), pipe.d_frame_src_mut(), pipe.d_count_frame());
            pipe.QueueCountsReadback();
            CAPI_CUDA(cudaStreamSynchronize(stream));
            total = pipe.h_counts()[1];
            const size_t k = std::min<size_t>(cap, (size_t) total);
            CAPI_CUDA(cudaMemcpy(out_indices, pipe.d_frame_src(), sizeof(uint32_t) * k, cudaMemcpyDeviceToHost));
        }
        cudaStreamDestroy(stream);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : total;
}
int64_t cticp_adaptive_sample_indices(int device, const cticp_adaptive_options *options, const double *xyz,
                                      size_t stride_bytes, size_t n, uint32_t *out_indices, size_t cap) {
    int64_t total = 0;
    int rc = Guard([&] {
        RequireDevice(device);
        if (n == 0 || !options) return (int) CTICP_OK;
        cudaStream_t stream;
        CAPI_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        {
            FramePipeline pipe(n, stream);
            float4 *stage = pipe.Staging(), *stage_lo = pipe.StagingLo();
            for (size_t i = 0; i < n; ++i) {
                const double *p = reinterpret_cast<const double *>(reinterpret_cast<const char *>(xyz) + stride_bytes * i);
                stage[i] = make_float4((float) p[0], (float) p[1], (float) p[2], 0.f);
                stage_lo[i] = make_float4((float) (p[0] - (double) stage[i].x), (float) (p[1] - (double) stage[i].y),
                                          (float) (p[2] - (double) stage[i].z), 0.f);
            }
            pipe.Upload(n);
            pipe.UploadLo(n);
            pipe.AdaptiveSelect(*options, pipe.d_raw(), pipe.d_raw_lo(), nullptr, pipe.d_count_n(), n, pipe.d_frame_mut(),
                                pipe.d_frame_lo_mut(), pipe.d_frame_src_mut(), pipe.d_count_frame());
            pipe.QueueCountsReadback();
            CAPI_CUDA(cudaStreamSynchronize(stream));
            total = pipe.h_counts()[1];
            const size_t k = std::min<size_t>(cap, (size_t) total);
            CAPI_CUDA(cudaMemcpy(out_indices, pipe.d_frame_src(), sizeof(uint32_t) * k, cudaMemcpyDeviceToHost));
        }
        cudaStreamDestroy(stream);
        return (int) CTICP_OK;
    });
    return rc < 0 ? rc : total;
}
int cticp_permutation(uint64_t seed, uint64_t counter, uint32_t n, uint32_t *out_perm) {
    // pure integer bijection (same __host__ __device__ code the kernels run): no device needed
    const Perm p = perm_make(seed, counter, n ? n : 1);
    for (uint32_t i = 0; i < n; ++i) out_perm[i] = perm_apply(p, i);
    return CTICP_OK;
}

int cticp_nccl_unique_id(void *out_128_bytes);   // nccl_shard.cu

}  // extern "C"
