/*
 * cticp.h — C ABI of the B200-native CT-ICP registration engine.
 *
 * This is the drop-in boundary underneath the C++ facade `ct_icp::Odometry`
 * (ct_icp_b200/include/ct_icp/odometry.h). Plain pointers and sizes only; no
 * C++/torch/Eigen types. Every entry point names the reference interface it
 * replaces (paths relative to the upstream tree, jedeschaud/ct_icp @ d467813).
 *
 * Conventions
 *   - return value: CTICP_OK (0) or a negative cticp_status; the message of the
 *     last failure is available through cticp_last_error().
 *   - quaternions are stored (x, y, z, w) like Eigen::Quaterniond::coeffs().
 *   - one handle owns one CUDA device context + stream; a handle is NOT
 *     re-entrant (same rule as the reference: callers serialise, see
 *     ros/catkin_ws/ct_icp_odometry/src/ct_icp_odometry_node.cxx:67).
 *   - input clouds are borrowed for the duration of the call only.
 *   - there is NO CPU fallback: cticp_create fails with CTICP_ERR_NO_DEVICE
 *     when no sm_100 device is usable.
 *   - ingest precision: a scan is kept on the device as (x, y, z, alpha) in
 *     fp32 — what LiDAR drivers emit (KITTI .bin, PointCloud2 FLOAT32) — and all
 *     geometry is evaluated in fp64 from there. The reference reads the scan
 *     through double-converting views (src/ct_icp/odometry.cpp:335-336), so for
 *     FLOAT32 sources the two agree exactly. FLOAT64 coordinates that fp32
 *     cannot hold travel with a second fp32 plane of residuals (value - fp32(value);
 *     hi + lo reproduces the double to ~2^-48 relative), uploaded only for such
 *     scans: the samplers then see the same voxel for every point as the
 *     reference does and the sample sets are identical
 *     (tests/test_gpu_parity_r2.py::test_fp64_scan_coordinates_and_timestamps).
 *     With FLOAT32 coordinates and wider timestamps alpha is rounded to fp32
 *     (<= 6e-8 of the sweep: <= 1e-6 m at 15 m/s); the timestamps returned in
 *     cticp_wpoint records are rebuilt from alpha.
 *   - multi-GPU (cticp_odometry_enable_sharding): ONE driving thread per rank —
 *     every exchange is a device-side rendezvous that needs all ranks' kernels in
 *     flight at once, so one host thread driving two handles in turn deadlocks
 *     until the exchange times out (CTICP_PEER_TIMEOUT_MS, default 30 s).
 */
#ifndef CTICP_H
#define CTICP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTICP_ABI_VERSION 1
#define CTICP_MAX_RESOLUTIONS 8

typedef enum cticp_status {
    CTICP_OK = 0,
    CTICP_ERR_INVALID_ARGUMENT = -1,
    CTICP_ERR_NO_DEVICE = -2,
    CTICP_ERR_CUDA = -3,
    CTICP_ERR_CAPACITY = -4,      /* a device table / block pool is full */
    CTICP_ERR_TIMESTAMP = -5,     /* reference: CHECK in TPose::InterpolatePose, include/SlamCore/types.h:456 */
    CTICP_ERR_UNSUPPORTED = -6,   /* option combination outside the built hot path */
    CTICP_ERR_NCCL = -7,
    CTICP_ERR_INTERNAL = -8,
    CTICP_ERR_CALLBACK = -9       /* a registered callback returned 0 (reference: CHECK, src/ct_icp/odometry.cpp:748) */
} cticp_status;

/* ---- enums mirroring the reference (same numeric order) ------------------------------------------------ */
/* include/ct_icp/ct_icp.h:35-39 */
/* scalar types of interleaved point records = sensor_msgs/PointField datatype codes
 * (ros/roscore/src/pc2_conversion.cxx:6-27, slam::PROPERTY_TYPE) */
enum { CTICP_DTYPE_INT8 = 1, CTICP_DTYPE_UINT8 = 2, CTICP_DTYPE_INT16 = 3, CTICP_DTYPE_UINT16 = 4,
       CTICP_DTYPE_INT32 = 5, CTICP_DTYPE_UINT32 = 6, CTICP_DTYPE_FLOAT32 = 7, CTICP_DTYPE_FLOAT64 = 8 };
enum { CTICP_SOLVER_GN = 0, CTICP_SOLVER_CERES = 1, CTICP_SOLVER_ROBUST = 2 };
/* include/ct_icp/ct_icp.h:41-47 */
enum { CTICP_LOSS_STANDARD = 0, CTICP_LOSS_CAUCHY = 1, CTICP_LOSS_HUBER = 2, CTICP_LOSS_TOLERANT = 3,
       CTICP_LOSS_TRUNCATED = 4 };
/* include/ct_icp/ct_icp.h:49-53 */
enum { CTICP_WEIGHT_PLANARITY = 0, CTICP_WEIGHT_NEIGHBORHOOD = 1, CTICP_WEIGHT_ALL = 2 };
/* include/ct_icp/cost_functions.h:17-20 (POSE_PARAMETRIZATION) */
enum { CTICP_PARAM_SIMPLE = 0, CTICP_PARAM_CONTINUOUS_TIME = 1 };
/* include/ct_icp/cost_functions.h:22-27 (ICP_DISTANCE) */
enum { CTICP_DIST_POINT_TO_PLANE = 0, CTICP_DIST_POINT_TO_POINT = 1, CTICP_DIST_POINT_TO_LINE = 2,
       CTICP_DIST_POINT_TO_DISTRIBUTION = 3 };
/* include/ct_icp/odometry.h:16-21 (MOTION_COMPENSATION) */
enum { CTICP_MC_NONE = 0, CTICP_MC_CONSTANT_VELOCITY = 1, CTICP_MC_ITERATIVE = 2, CTICP_MC_CONTINUOUS = 3 };
/* include/ct_icp/odometry.h:23-26 (INITIALIZATION) */
enum { CTICP_INIT_NONE = 0, CTICP_INIT_CONSTANT_VELOCITY = 1 };
/* include/ct_icp/odometry.h:27-31 (sampling::SAMPLING_OPTION) */
enum { CTICP_SAMPLING_NONE = 0, CTICP_SAMPLING_GRID = 1, CTICP_SAMPLING_ADAPTIVE = 2 };
/* include/ct_icp/motion_model.h:36-39 */
enum { CTICP_MM_CONSTANT_VELOCITY = 0, CTICP_MM_SMALL_VELOCITY = 1 };

/* ---- option PODs ------------------------------------------------------------------------------------------ */

/* ct_icp::CTICPOptions, include/ct_icp/ct_icp.h:56-153 (defaults: cticp_default_icp_options) */
typedef struct cticp_icp_options {
    int32_t num_iters_icp;
    int32_t parametrization;
    int32_t distance;
    int32_t solver;
    int32_t max_num_residuals;
    int32_t min_num_residuals;
    int32_t weighting_scheme;
    int32_t max_number_neighbors;
    int32_t min_number_neighbors;
    int32_t threshold_voxel_occupancy;
    int32_t num_closest_neighbors;
    int32_t point_to_plane_with_distortion;
    int32_t loss_function;
    int32_t ls_max_num_iters;
    int32_t ls_num_threads;
    int32_t debug_print;
    double weight_alpha;
    double weight_neighborhood;
    double power_planarity;
    double threshold_orientation_norm;
    double threshold_translation_norm;
    double ls_sigma;
    double ls_tolerant_min_threshold;
    double max_dist_to_plane_ct_icp;
    /* ROBUST solver params (include/ct_icp/ct_icp.h:133-141) */
    double threshold_linearity;
    double threshold_planarity;
    double weight_point_to_point;
    double outlier_distance;
    int32_t use_barycenter;
    int32_t use_lines;             /* ct_icp.h:140 (default true; not settable from the reference's YAML) */
} cticp_icp_options;

/* ct_icp::MultipleResolutionVoxelMap::ResolutionParam / Options, include/ct_icp/map.h:109-134 */
typedef struct cticp_resolution_param {
    double resolution;
    double min_distance_between_points;
    int32_t max_num_points;
    int32_t _pad0;
} cticp_resolution_param;

typedef struct cticp_map_options {
    int32_t num_resolutions;
    int32_t select_valid_normals_direction;
    int32_t max_frames_to_keep;
    int32_t _pad0;
    double default_radius;
    cticp_resolution_param resolutions[CTICP_MAX_RESOLUTIONS];
    /* device sizing (new; not in the reference): 0 = pick from defaults */
    uint64_t capacity_voxels;      /* slots per resolution (power of two is taken) */
} cticp_map_options;

/* ct_icp::INeighborStrategyOptions + DefaultNearestNeighborStrategy::Options + DistanceBasedStrategy::Options,
 * include/ct_icp/neighborhood_strategy.h:37-55, 60-85, 95-146. The strategy is consulted by solver CERES only
 * (src/ct_icp/ct_icp.cpp:571); GN and ROBUST search with the map's default radius. */
enum { CTICP_STRATEGY_NEAREST_NEIGHBOR = 0, CTICP_STRATEGY_DISTANCE_BASED = 1 };
typedef struct cticp_strategy_options {
    int32_t type;                  /* CTICP_STRATEGY_* */
    int32_t max_num_neighbors;
    int32_t min_num_neighbors;
    int32_t _pad0;
    /* DISTANCE_BASED_STRATEGY (:113-119): search radius grows with the keypoint's range; the map's per-point
     * normals reject neighbors whose surface faces away from the sensor (map.h:482-490) */
    double distance_max;
    double radius_min;
    double radius_max;
    double exponent;
} cticp_strategy_options;

/* ct_icp::PreviousFrameMotionModel::Options, include/ct_icp/motion_model.h:42-58 */
typedef struct cticp_motion_model_options {
    int32_t model;
    int32_t log_if_invalid;
    double beta_location_consistency;
    double beta_constant_velocity;
    double beta_small_velocity;
    double beta_orientation_consistency;
    double threshold_orientation_deg;
    double threshold_translation_diff;
} cticp_motion_model_options;

/* ct_icp::AdaptiveGridSamplingOptions, include/ct_icp/algorithm/sampling.h:14-27 */
#define CTICP_MAX_ADAPTIVE_BANDS 8
typedef struct cticp_adaptive_options {
    int32_t num_points_per_voxel;      /* only 1 is built */
    int32_t max_num_points;
    int32_t num_bands;                 /* entries of distance_voxel_size */
    int32_t _pad0;
    double distance[CTICP_MAX_ADAPTIVE_BANDS];     /* .first  : distance to the sensor */
    double voxel_size[CTICP_MAX_ADAPTIVE_BANDS];   /* .second : sampling voxel of the band starting there */
} cticp_adaptive_options;

/* ct_icp::OdometryOptions, include/ct_icp/odometry.h:32-157 */
typedef struct cticp_odometry_options {
    cticp_icp_options ct_icp_options;
    cticp_map_options map_options;
    cticp_strategy_options neighborhood_strategy;
    cticp_motion_model_options default_motion_model;
    int32_t motion_compensation;
    int32_t initialization;
    int32_t init_num_frames;
    int32_t max_num_keypoints;
    int32_t sampling;
    int32_t quit_on_error;
    int32_t robust_minimal_level;
    int32_t robust_registration;
    int32_t robust_fail_early;
    int32_t robust_num_attempts;
    int32_t robust_num_attempts_when_rotation;
    int32_t robust_max_voxel_neighborhood;
    int32_t always_insert;
    int32_t do_no_insert;
    int32_t debug_print;
    int32_t with_default_motion_model;
    double init_voxel_size;
    double init_sample_voxel_size;
    double sample_voxel_size;
    double voxel_size;
    double max_distance;
    double distance_error_threshold;
    double orientation_error_threshold;
    double robust_full_voxel_threshold;
    double robust_empty_voxel_threshold;
    double robust_neighborhood_min_dist;
    double robust_neighborhood_min_orientation;
    double robust_relative_trans_threshold;
    double robust_threshold_ego_orientation;
    double robust_threshold_relative_orientation;
    double insertion_ego_rotation_threshold;
    double insertion_threshold_frames_skipped;
    double insertion_cum_distance_threshold;
    double insertion_cum_orientation_threshold;
    /* order contract (new): seed of the counter-based permutations that stand in for
     * std::shuffle(…, std::mt19937_64 g_) at src/ct_icp/odometry.cpp:349,361,550 */
    uint64_t shuffle_seed;
    /* device sizing (new): upper bound on points per scan; 0 = 524288 */
    uint64_t max_points_per_frame;
    cticp_adaptive_options adaptive_options;   /* sampling == ADAPTIVE */
} cticp_odometry_options;

/* ---- value PODs ------------------------------------------------------------------------------------------- */

/* slam::TPose<double>, include/SlamCore/types.h:162-274 */
typedef struct cticp_pose {
    double quat[4];                /* x, y, z, w */
    double tr[3];
    double ref_timestamp;
    double dest_timestamp;
    uint32_t ref_frame_id;
    uint32_t dest_frame_id;
} cticp_pose;

/* ct_icp::TrajectoryFrame, include/ct_icp/types.h:31-61 */
typedef struct cticp_frame {
    cticp_pose begin_pose;
    cticp_pose end_pose;
} cticp_frame;

/* slam::WPoint3D, include/SlamCore/types.h:35-60 (same 64-byte layout: raw xyz, t, world xyz, index_frame) */
typedef struct cticp_wpoint {
    double raw[3];
    double timestamp;
    double world[3];
    uint32_t index_frame;
    uint32_t _pad0;
} cticp_wpoint;

/* ct_icp::ICPSummary, include/ct_icp/ct_icp.h:155-169 */
typedef struct cticp_icp_summary {
    int32_t success;
    int32_t num_residuals_used;
    int32_t num_iters;
    int32_t _pad0;
    double duration_total;
    double duration_init;
    double avg_duration_iter;
    double avg_duration_neighborhood;
    double avg_duration_solve;
} cticp_icp_summary;

/* ct_icp::Odometry::RegistrationSummary, include/ct_icp/odometry.h:163-199.
 * The three point vectors are fetched on demand with cticp_odometry_get_points. */
typedef struct cticp_summary {
    cticp_frame frame;
    cticp_frame initial_frame;
    cticp_icp_summary icp_summary;
    int32_t sample_size;
    int32_t number_of_residuals;
    int32_t robust_level;
    int32_t success;
    int32_t points_added;
    int32_t number_of_attempts;
    double distance_correction;
    double relative_distance;
    double relative_orientation;
    double ego_orientation;
    uint64_t num_corrected_points;       /* F: points of the sub-sampled frame */
    uint64_t num_all_corrected_points;   /* N: points of the input scan */
    uint64_t num_keypoints;              /* K */
    /* logged_values (src/ct_icp/odometry.cpp:495-513), milliseconds */
    double odometry_total;
    double odometry_initialization;
    double odometry_try_register;
    double odometry_duration_sampling;
    double odometry_map_update;
    double odometry_transform;
    char error_message[256];
} cticp_summary;

enum { CTICP_POINTS_CORRECTED = 0, CTICP_POINTS_ALL_CORRECTED = 1, CTICP_POINTS_KEYPOINTS = 2 };

typedef struct cticp_odometry cticp_odometry;   /* opaque: replaces ct_icp::Odometry */
typedef struct cticp_map cticp_map;             /* opaque: replaces ct_icp::MultipleResolutionVoxelMap */

/* ---- defaults & profiles ---------------------------------------------------------------------------------- */
uint32_t cticp_abi_version(void);
const char *cticp_last_error(void);                                   /* thread-local */

void cticp_default_icp_options(cticp_icp_options *out);               /* include/ct_icp/ct_icp.h:60-152 */
void cticp_default_map_options(cticp_map_options *out);               /* include/ct_icp/map.h:115-125 */
void cticp_default_odometry_options(cticp_odometry_options *out);     /* include/ct_icp/odometry.h:37-157 */
void cticp_legacy_map_options(cticp_map_options *out, double size_voxel_map, int max_num_points_in_voxel,
                              double min_distance_points);            /* src/ct_icp/map.cpp:13-29 */
void cticp_profile_default_driving(cticp_odometry_options *out);      /* src/ct_icp/odometry.cpp:30-36 */
void cticp_profile_robust_driving(cticp_odometry_options *out);       /* src/ct_icp/odometry.cpp:39-89 */
void cticp_profile_robust_outdoor_low_inertia(cticp_odometry_options *out); /* src/ct_icp/odometry.cpp:92-151 */

/* ---- Odometry (L4 boundary) ------------------------------------------------------------------------------- */

/* ct_icp::Odometry::Odometry(const OdometryOptions&), src/ct_icp/odometry.cpp:697-734 */
int cticp_odometry_create(const cticp_odometry_options *options, int device, cticp_odometry **out);
void cticp_odometry_destroy(cticp_odometry *h);

/* ct_icp::Odometry::RegisterFrame(const slam::PointCloud&, frame_id_t, AMotionModel*), src/ct_icp/odometry.cpp:199-214
 * and RegisterFrameWithEstimate (:217-236) when initial_estimate != NULL.
 * xyz / t are strided HOST arrays (stride in bytes), the layout RegisterFrame reads through
 * XYZConst<double>() / TimestampsProxy<double>() (src/ct_icp/odometry.cpp:335-336). */
int cticp_odometry_register_frame(cticp_odometry *h,
                                  const double *xyz, size_t xyz_stride_bytes,
                                  const double *t, size_t t_stride_bytes,
                                  size_t n, uint32_t frame_id,
                                  const cticp_frame *initial_estimate,
                                  cticp_summary *out_summary);

/* The AMotionModel* argument of the RegisterFrame overloads (include/ct_icp/odometry.h:231-248). The reference's only
 * concrete model is PreviousFrameMotionModel (include/ct_icp/motion_model.h:35-78): its options and the previous frame it
 * was updated with. NULL = the reference's nullptr (the odometry's own default model when with_default_motion_model). */
typedef struct cticp_motion_prior {
    cticp_motion_model_options options;
    cticp_frame previous_frame;
} cticp_motion_prior;
int cticp_odometry_register_frame_ex(cticp_odometry *h,
                                     const double *xyz, size_t xyz_stride_bytes,
                                     const double *t, size_t t_stride_bytes,
                                     size_t n, uint32_t frame_id,
                                     const cticp_frame *initial_estimate,      /* nullable */
                                     const cticp_motion_prior *motion_model,   /* nullable */
                                     cticp_summary *out_summary);

/* ct_icp::Odometry::RegisterCallback (include/ct_icp/odometry.h:260, src/ct_icp/odometry.cpp:737-750): ONE hook per
 * handle, called on the registering thread at the reference's three events; inside it the caller may use
 * cticp_odometry_get_points (frame / keypoints with the pose pair of that moment). Returning 0 aborts the
 * registration with CTICP_ERR_CALLBACK. fn == NULL removes the hook. */
enum { CTICP_EVENT_BEFORE_ITERATION = 0, CTICP_EVENT_ITERATION_COMPLETED = 1, CTICP_EVENT_FINISHED_REGISTRATION = 2 };
typedef int (*cticp_event_fn)(int event, void *user);
int cticp_odometry_set_callback(cticp_odometry *h, cticp_event_fn fn, void *user);

/* An interleaved point buffer described like a sensor_msgs/PointCloud2 (one record every point_step bytes; field
 * "x" at xyz_offset with y and z following contiguously in the same scalar type — the "vertex" element that
 * SchemaBuilderFromCloud2 builds, ros/roscore/src/pc2_conversion.cxx:73-80 — and one timestamp scalar at t_offset).
 * It is the zero-copy input of the ROS node (ROSCloud2ToSlamPointCloudShallow, pc2_conversion.cxx:86-96 →
 * RegisterFrame(const slam::PointCloud&), src/ct_icp/odometry.cpp:199-214): the engine reads the records in place
 * and converts each scalar with static_cast<double>, as the reference's proxy views do
 * (include/SlamCore/data/view.h:99-120). Records need no alignment. */
typedef struct cticp_cloud_view {
    const void *data;
    uint64_t num_points;           /* width * height */
    uint32_t point_step;
    uint32_t xyz_offset;
    int32_t xyz_dtype;             /* CTICP_DTYPE_FLOAT32 or CTICP_DTYPE_FLOAT64 */
    uint32_t t_offset;
    int32_t t_dtype;               /* any CTICP_DTYPE_* */
    int32_t _pad0;
} cticp_cloud_view;

/* RegisterFrame(const slam::PointCloud&, frame_id) / RegisterFrameWithEstimate on a record buffer. */
int cticp_odometry_register_cloud(cticp_odometry *h, const cticp_cloud_view *cloud, uint32_t frame_id,
                                  const cticp_frame *initial_estimate, cticp_summary *out_summary);
/* cticp_odometry_stage_frame on a record buffer. */
int64_t cticp_odometry_stage_cloud(cticp_odometry *h, const cticp_cloud_view *cloud);

/* Egress in the caller's record layout (what the ROS node builds from summary.corrected_points / keypoints for its
 * publishers: pcl::PointCloud<slam::XYZTPoint>, ct_icp_odometry_node.cxx:228-262): writes world (world != 0) or raw
 * x,y,z and, when t_dtype != 0, the timestamp of min(capacity_points, count) points. Returns the count. */
typedef struct cticp_cloud_sink {
    void *data;
    uint64_t capacity_points;
    uint32_t point_step;
    uint32_t xyz_offset;
    int32_t xyz_dtype;             /* CTICP_DTYPE_FLOAT32 or CTICP_DTYPE_FLOAT64 */
    uint32_t t_offset;
    int32_t t_dtype;               /* 0 = no timestamp; else CTICP_DTYPE_FLOAT32 / CTICP_DTYPE_FLOAT64 */
    int32_t world;
} cticp_cloud_sink;
int64_t cticp_odometry_write_points(cticp_odometry *h, int which, const cticp_cloud_sink *sink);

/* RegistrationSummary::{corrected_points, all_corrected_points, keypoints}, include/ct_icp/odometry.h:187-191.
 * Copies min(cap, count) points device->host; returns the count or a negative status. */
int64_t cticp_odometry_get_points(cticp_odometry *h, int which, cticp_wpoint *dst, size_t cap);
/* RegistrationSummary returns its three point vectors BY VALUE from every RegisterFrame (src/ct_icp/odometry.cpp:462-486,
 * 597). mask: bit CTICP_POINTS_* set = that vector is produced eagerly by every following cticp_odometry_register_* call
 * (world coordinates transformed and copied to pinned host memory on a second stream, next to the map update), so the
 * cticp_odometry_get_points that follows only assembles the 64-byte records. 0 (default) = on demand. */
int cticp_odometry_set_summary_points(cticp_odometry *h, int mask);

/* ct_icp::Odometry::Trajectory(), src/ct_icp/odometry.cpp:687-689 */
int64_t cticp_odometry_trajectory(cticp_odometry *h, cticp_frame *dst, size_t cap);
/* ct_icp::Odometry::MapSize(), src/ct_icp/odometry.cpp:156-158 */
int64_t cticp_odometry_map_size(cticp_odometry *h);
/* ct_icp::Odometry::GetMapPointCloud(), src/ct_icp/odometry.cpp:692-694 → xyz triples */
int64_t cticp_odometry_map_points(cticp_odometry *h, double *dst_xyz, size_t cap_points);
/* ct_icp::Odometry::Reset(), src/ct_icp/odometry.cpp:956-965 */
int cticp_odometry_reset(cticp_odometry *h);
/* ct_icp::Odometry::Reset(const OdometryOptions&), include/ct_icp/odometry.h:269: same handle, new options (new map) */
int cticp_odometry_reset_options(cticp_odometry *h, const cticp_odometry_options *options);
/* ct_icp::Odometry::GetMapPointer(), src/ct_icp/odometry.cpp:991-993 (borrowed; owned by the odometry) */
cticp_map *cticp_odometry_map(cticp_odometry *h);

/* multi-GPU (new; SURVEY §8e): keypoints sharded rank/world, one exchange (sum over ranks) of JTJ/JTr per GN
 * iteration / LM evaluation. unique_id is the 128-byte ncclUniqueId produced by cticp_nccl_unique_id on rank 0 and
 * broadcast by the caller; NCCL bootstraps NVLink peer mailboxes (CUDA IPC) through which the ICP kernels exchange
 * the accumulators themselves, and stays as the fallback (ncclAllReduce per exchange) where peers cannot be mapped. */
int cticp_nccl_unique_id(void *out_128_bytes);
int cticp_odometry_enable_sharding(cticp_odometry *h, const void *unique_id_128_bytes, int rank, int world);
/* 0 = not sharded, 1 = exchange through ncclAllReduce, 2 = in-kernel exchange over peer mailboxes */
int cticp_odometry_sharding_mode(cticp_odometry *h);

/* ---- checkpoint / resume (new; the reference has no checkpoint of odometry state, SURVEY §5) ---------------
 * A blob holds everything that influences the frames to come: the effective options (after the motion-compensation
 * overrides of the constructor), the trajectory, the robust-registration ladder, the insertion tracker, the default
 * motion model, the keypoint-count hint of the ICP kernels, and the device map (voxel keys, fp32 point runs, per-voxel
 * normals, begin position of every inserted frame). A run saved after frame k and loaded into a new handle produces the
 * same bits for every later frame as the run that never stopped. The point vectors of the last registered frame are
 * not state: after a load the get_points / write_points calls answer as on a new handle.
 * Layout (little-endian, sections 8-byte aligned; DESIGN.md §9 has every field):
 *   odometry: "CTICPODO", u32 version, u32 sizeof(cticp_odometry_options), u64 total_bytes, u64 checksum, options,
 *             host-state record, cticp_frame trajectory[T], one map blob
 *   map:      "CTICPMAP", u32 version, u32 num_levels, u64 total_bytes, u64 checksum, u32 has_normals, u32 0,
 *             u64 frame_count, [f64 frame_origins[3 * frame_count]], per level: f64 resolution, f64 min_distance,
 *             i32 max_num_points, i32 0, u64 V, u64 P, u64 keys[V] (ascending), u32 counts[V] (padded to 8 bytes),
 *             float4 points[P], [f64 normals[4 * V]]
 *   checksum: FNV-1a 64 over bytes [32, total_bytes) read as u64 words (guards against truncation and corruption).
 * Blobs are canonical: voxels in ascending packed-key order, points in insertion order inside a voxel, so saving the
 * same state twice gives the same bytes.
 * save: returns the blob size and writes only when cap >= size; waits for the work in flight, changes nothing.
 * load: replaces the handle's whole state (also after frames were registered). Options must be equal except
 * map_options.capacity_voxels and max_points_per_frame (CTICP_ERR_INVALID_ARGUMENT names the first differing field);
 * the tables are sized for the loaded map. Any rejected blob leaves the handle untouched. A sharded handle can save,
 * but its load fails with CTICP_ERR_UNSUPPORTED. */
int64_t cticp_odometry_save_state(cticp_odometry *h, void *dst, size_t cap);
int cticp_odometry_load_state(cticp_odometry *h, const void *src, size_t size);
/* the options stored in an odometry blob (no device needed): create the handle to load the blob into from them */
int cticp_odometry_state_options(const void *src, size_t size, cticp_odometry_options *out);

/* device timing of the last register_frame (CUDA events on the handle's stream), milliseconds */
typedef struct cticp_device_timing {
    double total_ms;
    double ingest_ms;        /* H2D + sub-sampling + keypoint sampling */
    double icp_ms;           /* all ICP iterations (gather kernel + solve) */
    double gather_ms;        /* neighbor-gather/residual kernel only, summed over iterations */
    double map_update_ms;    /* transform + evict + insert */
    int32_t icp_iterations;
    int32_t kernel_launches;
    uint64_t gather_keypoint_iterations;   /* Σ over iterations of keypoints processed */
    uint64_t gather_stencil_points;        /* Σ S: map points found inside the stencils */
    uint64_t gather_stencil_voxels;        /* Σ (2r+1)^3 probes */
    uint64_t h2d_bytes;                    /* host→device bytes copied by the call (scan + state) */
    uint64_t d2h_bytes;                    /* device→host bytes copied by the call (poses, counters) */
    int32_t gather_launches;               /* launches of the neighbor-gather kernel */
    int32_t _pad0;
} cticp_device_timing;
int cticp_odometry_last_timing(cticp_odometry *h, cticp_device_timing *out);

/* Device-resident input (new): a scan can be packed and copied to HBM ahead of time (e.g. by a decoder that
 * already runs on the GPU) and registered later without any host→device traffic for the points.
 * cticp_odometry_stage_frame returns a slot id >= 0; slots live until cticp_odometry_clear_staged. */
int64_t cticp_odometry_stage_frame(cticp_odometry *h, const double *xyz, size_t xyz_stride_bytes, const double *t,
                                   size_t t_stride_bytes, size_t n);
int cticp_odometry_register_staged(cticp_odometry *h, int64_t slot, uint32_t frame_id, cticp_summary *out_summary);
int cticp_odometry_clear_staged(cticp_odometry *h);
/* CUDA-event stopwatch on the handle's stream (the stream every kernel of this handle is launched on) */
int cticp_odometry_timer_start(cticp_odometry *h);
int cticp_odometry_timer_stop(cticp_odometry *h, double *elapsed_ms);   /* synchronises */
/* per-launch CUDA-event timing of the gather kernel (adds two event records per ICP iteration) */
int cticp_odometry_set_gather_timing(cticp_odometry *h, int on);
/* writes `bytes` of device memory (> L2 size flushes the L2) on the handle's stream */
int cticp_odometry_flush_l2(cticp_odometry *h, size_t bytes);

/* ---- Map (L2 boundary; used directly by the parity tests) ---------------------------------------------- */

/* MultipleResolutionVoxelMap(const Options&), include/ct_icp/map.h:136-138 */
int cticp_map_create(const cticp_map_options *options, int device, cticp_map **out);
void cticp_map_destroy(cticp_map *m);
/* InsertPointCloud (world points, given order), include/ct_icp/map.h:153-254,261-293 */
int cticp_map_insert(cticp_map *m, const double *xyz, size_t stride_bytes, size_t n);
/* InsertPointCloud(pointcloud, frame_poses, ...) where the begin pose of the source frame matters: per-voxel normals
 * are oriented towards `origin` = frame_poses.front().tr (include/ct_icp/map.h:211-235). cticp_map_insert is the same
 * with origin = (0, 0, 0). */
int cticp_map_insert_from(cticp_map *m, const double *xyz, size_t stride_bytes, size_t n, const double origin[3]);
/* RemoveElementsFarFromLocation, include/ct_icp/map.h:305-322 */
int cticp_map_remove_far(cticp_map *m, const double location[3], double distance);
/* NumPoints(), include/ct_icp/map.h:345 (resolution 0) ; num points of any resolution with map_idx */
int64_t cticp_map_num_points(cticp_map *m, int map_idx);
int64_t cticp_map_num_voxels(cticp_map *m, int map_idx);
/* GetMapPoints(map_idx), include/ct_icp/map.h:354-376: xyz + int32 voxel coords per point (either may be NULL) */
int64_t cticp_map_export(cticp_map *m, int map_idx, double *dst_xyz, int32_t *dst_voxel, size_t cap_points);
/* ComputeNeighborhoods(queries, max_num_neighbors), include/ct_icp/map.h:532-540 (default radius, no normal filter).
 * out_points: n × max_num_neighbors × 3 (farthest first, like RadiusSearchInPlace :508-513), out_counts: n */
int cticp_map_compute_neighborhoods(cticp_map *m, const double *queries_xyz, size_t n, int max_num_neighbors,
                                    double *out_points, int32_t *out_counts);
/* ComputeNeighborhoods(queries, radiuses, max_num_neighbors, nearest_neighbors = true, sensor_location),
 * include/ct_icp/map.h:434-447 → RadiusSearchInPlace :449-514: one radius per query (it selects the resolution and the
 * stencil, :416-432); when sensor_location != NULL and the map's select_valid_normals_direction is set, stored points
 * whose oriented normal faces away from the sensor are skipped (:482-490). Output layout as above. */
int cticp_map_radius_search(cticp_map *m, const double *queries_xyz, const double *radiuses, size_t n,
                            int max_num_neighbors, const double *sensor_location, double *out_points,
                            int32_t *out_counts);
/* ClearMap(), include/ct_icp/map.h:296 */
int cticp_map_clear(cticp_map *m);
/* the map blob above, alone (new). load requires equal resolutions, max_num_points, min_distance_between_points and
 * the same choice of keeping per-voxel normals (select_valid_normals_direction); capacity may differ. A map that
 * belongs to an odometry can be saved but not loaded (CTICP_ERR_UNSUPPORTED): load the odometry's state instead. */
int64_t cticp_map_save(cticp_map *m, void *dst, size_t cap);
int cticp_map_load(cticp_map *m, const void *src, size_t size);

/* ---- Registration (L3 boundary) ------------------------------------------------------------------------- */

/* CT_ICP_Registration::Register(map, keypoints, frame, motion_model, strategy), src/ct_icp/ct_icp.cpp:1026-1037.
 * keypoints[i].world is rewritten (as the reference does through the world_point proxy);
 * frame is in/out; previous_frame (nullable) stands for the PreviousFrameMotionModel state and
 * motion_options for its Options (src/ct_icp/motion_model.cpp:12-61, ct_icp.cpp:885-910). */
int cticp_icp_register(cticp_map *m, const cticp_icp_options *options,
                       const cticp_strategy_options *strategy,
                       cticp_wpoint *keypoints, size_t n,
                       cticp_frame *frame,
                       const cticp_frame *previous_frame,
                       const cticp_motion_model_options *motion_options,
                       cticp_icp_summary *out_summary);

/* Debug tap for parity tests: normal equations of ONE Gauss-Newton linearisation at `frame`
 * (A 12×12 row-major AFTER the 1/n normalisation and regularisers of ct_icp.cpp:877-910, b 12, n used). */
int cticp_icp_gn_normal_equations(cticp_map *m, const cticp_icp_options *options,
                                  const cticp_wpoint *keypoints, size_t n,
                                  const cticp_frame *frame,
                                  const cticp_frame *previous_frame,
                                  const cticp_motion_model_options *motion_options,
                                  double *out_A144, double *out_b12, int32_t *out_num_used);

/* ---- Sampling (a3/a4) ------------------------------------------------------------------------------------ */

/* ct_icp::sub_sample_frame / grid_sampling, src/ct_icp/ct_icp.cpp:65-101, under the order contract
 * (first-seen per voxel of RAW coordinates in the given order; output in order of first appearance).
 * out_indices receives the indices kept; returns the count. */
int64_t cticp_grid_sample_indices(int device, const double *xyz, size_t stride_bytes, size_t n, double voxel_size,
                                  uint32_t *out_indices, size_t cap);
/* The counter-based permutation standing in for std::shuffle: out[perm(i)] = i semantics, see DESIGN.md */
int cticp_permutation(uint64_t seed, uint64_t counter, uint32_t n, uint32_t *out_perm);
/* ct_icp::AdaptiveSamplePointsInGrid, include/ct_icp/algorithm/sampling.h:55-110 (order contract: band by band, first
 * appearance inside a band). out_indices receives the indices kept; returns the count. */
int64_t cticp_adaptive_sample_indices(int device, const cticp_adaptive_options *options, const double *xyz,
                                      size_t stride_bytes, size_t n, uint32_t *out_indices, size_t cap);
void cticp_default_adaptive_options(cticp_adaptive_options *out);

#ifdef __cplusplus
}
#endif
#endif /* CTICP_H */
