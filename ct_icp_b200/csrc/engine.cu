// engine.cu — host orchestration of the B200-native odometry (see engine.h).
#include "engine.h"
#include "state_io.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include <emmintrin.h>
#include <xmmintrin.h>

#include <nvtx3/nvToolsExt.h>   // header-only: ranges are no-ops unless a profiler injects the NVTX library

namespace cticp {

#define CT_CUDA_CHECK(expr)                                                                              \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            throw CudaError(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                            std::to_string(__LINE__));                                                   \
    } while (0)

// NVTX range of one stage of RegisterFrame (ingest / sample / icp / map_update / egress): timelines of ncu / nsys-less tools
// attribute the launches to the stage that enqueued them
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

using hclock = std::chrono::steady_clock;

// ---- the tail of a plain registration, decided on the device (frame_policy.h) ------------------------------------------
// One warp. AssessRegistration (odometry.cpp:604-684, the branch without robust_registration) and UpdateMap's insertion
// policy (:903-925) on the registration state the ICP kernel left in HBM; the verdict goes to device memory (read by the
// speculative k_map_update_fused enqueued right behind) and to mapped pinned host memory, sequence number last.
__global__ void __launch_bounds__(32) k_frame_policy(const IcpState *__restrict__ st, const int *__restrict__ counts,
                                                     FramePolicyIn in, FrameVerdict *dv, FrameVerdict *hv) {
    __shared__ FrameVerdict v;
    const int lane = threadIdx.x;
    {
        const int *src = reinterpret_cast<const int *>(st);
        int *dst = reinterpret_cast<int *>(&v.state);
        for (int i = lane; i < (int) (sizeof(IcpState) / sizeof(int)); i += 32) dst[i] = __ldcg(src + i);
    }
    if (lane < 4) v.counts[lane] = __ldcg(counts + lane);
    __syncwarp();
    if (lane == 0) frame_policy_decide(v, in);
    __syncwarp();
    frame_verdict_publish(v, dv, hv, lane);
}
static double ms_since(hclock::time_point t0) {
    return std::chrono::duration<double, std::milli>(hclock::now() - t0).count();
}

HostPose PoseFromC(const cticp_pose &c) {
    HostPose p;
    p.pose.q = Q4{c.quat[0], c.quat[1], c.quat[2], c.quat[3]};
    p.pose.t = V3{c.tr[0], c.tr[1], c.tr[2]};
    p.ref_timestamp = c.ref_timestamp;
    p.dest_timestamp = c.dest_timestamp;
    p.ref_frame_id = c.ref_frame_id;
    p.dest_frame_id = c.dest_frame_id;
    return p;
}
cticp_pose PoseToC(const HostPose &p) {
    cticp_pose c;
    c.quat[0] = p.pose.q.x; c.quat[1] = p.pose.q.y; c.quat[2] = p.pose.q.z; c.quat[3] = p.pose.q.w;
    c.tr[0] = p.pose.t.x; c.tr[1] = p.pose.t.y; c.tr[2] = p.pose.t.z;
    c.ref_timestamp = p.ref_timestamp;
    c.dest_timestamp = p.dest_timestamp;
    c.ref_frame_id = p.ref_frame_id;
    c.dest_frame_id = p.dest_frame_id;
    return c;
}
HostFrame FrameFromC(const cticp_frame &c) { return HostFrame{PoseFromC(c.begin_pose), PoseFromC(c.end_pose)}; }
cticp_frame FrameToC(const HostFrame &f) { return cticp_frame{PoseToC(f.begin_pose), PoseToC(f.end_pose)}; }

// TPose::GetAlphaTimestamp, include/SlamCore/types.h:192-219 (incl. the "t > max → 0" quirk)
static double AlphaTimestamp(double t, double begin_ts, double end_ts) {
    const double mn = std::min(begin_ts, end_ts), mx = std::max(begin_ts, end_ts);
    if (mn > t) return 0.0;
    if (mx < t) return 0.0;
    if (mn == mx) return 1.0;
    return (t - mn) / (mx - mn);
}
static double EgoAngularDistance(const HostFrame &f) { return angular_distance_deg(f.begin_pose.pose.q, f.end_pose.pose.q); }

// ---------------------------------------------------------------------------------------------------------------
Engine::Engine(const cticp_odometry_options &options, int device) : options_(options), device_(device) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count)
        throw std::runtime_error("NO_DEVICE");
    CT_CUDA_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CT_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) throw std::runtime_error("NO_DEVICE: this build targets sm_100a (Blackwell B200) only");

    // Odometry::Odometry, odometry.cpp:697-734: motion_compensation overrides the ICP parametrisation
    switch (options_.motion_compensation) {
        case CTICP_MC_NONE:
        case CTICP_MC_CONSTANT_VELOCITY:   // ElasticICP does not compensate the motion
            options_.ct_icp_options.point_to_plane_with_distortion = 0;
            options_.ct_icp_options.distance = CTICP_DIST_POINT_TO_PLANE;
            options_.ct_icp_options.parametrization = CTICP_PARAM_SIMPLE;
            break;
        case CTICP_MC_ITERATIVE:           // … compensates the motion at each ICP iteration
            options_.ct_icp_options.point_to_plane_with_distortion = 1;
            options_.ct_icp_options.distance = CTICP_DIST_POINT_TO_PLANE;
            options_.ct_icp_options.parametrization = CTICP_PARAM_SIMPLE;
            break;
        case CTICP_MC_CONTINUOUS:          // … compensates continuously the motion
            options_.ct_icp_options.point_to_plane_with_distortion = 1;
            options_.ct_icp_options.parametrization = CTICP_PARAM_CONTINUOUS_TIME;
            options_.ct_icp_options.distance = CTICP_DIST_POINT_TO_PLANE;
            break;
        default:
            throw std::invalid_argument("unknown motion_compensation");
    }
    if (options_.sampling == CTICP_SAMPLING_ADAPTIVE && options_.adaptive_options.num_points_per_voxel != 1)
        throw UnsupportedError("sampling ADAPTIVE: only num_points_per_voxel == 1 is built");
    next_robust_level_ = options_.robust_minimal_level;
    if (const char *e = getenv("CTICP_FUSED_SAMPLING")) fused_sampling_ = atoi(e) != 0;
    if (const char *e = getenv("CTICP_FUSED_MAP_UPDATE")) fused_map_update_ = atoi(e) != 0;
    if (const char *e = getenv("CTICP_DEVICE_TAIL")) device_tail_ = atoi(e) != 0;
    if (const char *e = getenv("CTICP_TAIL_IN_KERNEL")) tail_in_kernel_ = atoi(e) != 0;

    {
        pool_ = std::make_unique<HostPool>(HostTeamSize(1));
    }
    CT_CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    // per-voxel normals are only read by the DistanceBasedStrategy's sensor-side filter (map.h:482-490)
    const bool with_normals = options_.map_options.select_valid_normals_direction &&
                              options_.neighborhood_strategy.type == CTICP_STRATEGY_DISTANCE_BASED;
    map_ = std::make_unique<DeviceMap>(options_.map_options, stream_, with_normals);
    const size_t max_pts = options_.max_points_per_frame ? (size_t) options_.max_points_per_frame : (size_t) 524288;
    pipe_ = std::make_unique<FramePipeline>(max_pts, stream_);
    icp_ = std::make_unique<IcpSolver>(stream_);
    CT_CUDA_CHECK(cudaMalloc(&d_state_, sizeof(IcpState)));
    CT_CUDA_CHECK(cudaMallocHost(&h_state_, sizeof(IcpState)));
    CT_CUDA_CHECK(cudaMalloc(&d_verdict_, sizeof(FrameVerdict)));
    CT_CUDA_CHECK(cudaMemsetAsync(d_verdict_, 0, sizeof(FrameVerdict), stream_));
    CT_CUDA_CHECK(cudaHostAlloc(&h_verdict_, sizeof(FrameVerdict), cudaHostAllocMapped));
    memset(h_verdict_, 0, sizeof(FrameVerdict));
    CT_CUDA_CHECK(cudaHostGetDevicePointer((void **) &h_verdict_dev_, h_verdict_, 0));
    CT_CUDA_CHECK(cudaStreamCreateWithFlags(&aux_stream_, cudaStreamNonBlocking));
    CT_CUDA_CHECK(cudaEventCreateWithFlags(&ev_state_up_, cudaEventDisableTiming));
    CT_CUDA_CHECK(cudaMalloc(&d_kp_world_, sizeof(double) * 3 * max_pts));
    for (auto &e : ev_) CT_CUDA_CHECK(cudaEventCreate(&e));
    for (auto &e : timer_ev_) CT_CUDA_CHECK(cudaEventCreate(&e));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
}

Engine::~Engine() {
    cudaSetDevice(device_);
    if (stream_) cudaStreamSynchronize(stream_);
    DestroySharding();
    icp_.reset();
    pipe_.reset();
    map_.reset();
    cudaFree(d_state_);
    cudaFreeHost(h_state_);
    cudaFree(d_verdict_);
    cudaFreeHost(h_verdict_);
    if (ev_state_up_) cudaEventDestroy(ev_state_up_);
    if (aux_stream_) cudaStreamDestroy(aux_stream_);
    cudaFree(d_kp_world_);
    for (auto &e : ev_) cudaEventDestroy(e);
    for (auto &e : timer_ev_) cudaEventDestroy(e);
    for (auto &sc : staged_) { cudaFree(sc.d_points); cudaFree(sc.d_lo); }
    cudaFree(d_flush_);
    for (int i = 0; i < 3; ++i) {
        cudaFreeHost(h_world_[i]);
        cudaFreeHost(h_src_[i]);
    }
    if (ev_egress_main_) cudaEventDestroy(ev_egress_main_);
    if (ev_egress_done_) cudaEventDestroy(ev_egress_done_);
    for (auto &e : ev_egress_chunk_)
        if (e) cudaEventDestroy(e);
    if (egress_stream_) cudaStreamDestroy(egress_stream_);
    if (stream_) cudaStreamDestroy(stream_);
}

void Engine::Reset() {   // odometry.cpp:956-965
    CT_CUDA_CHECK(cudaSetDevice(device_));
    trajectory_.clear();
    map_->Clear();
    registered_frames_ = 0;
    robust_num_consecutive_failures_ = 0;
    suspect_registration_error_ = false;
    next_robust_level_ = 0;
    tracker_ = {};
    default_motion_model_ = MotionModel();
    last_num_keypoints_ = 0;   // grid-size hint: keeps a reset run bit-identical to a fresh one
    last_all_world_valid_ = last_kp_world_valid_ = false;
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (egress_stream_) CT_CUDA_CHECK(cudaStreamSynchronize(egress_stream_));
    egress_pending_ = false;
    egress_valid_[0] = egress_valid_[1] = egress_valid_[2] = false;
    tail_event_valid_ = false;
    staging_in_flight_ = false;
}

int64_t Engine::SaveState(uint8_t *dst, size_t cap) {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    // the speculative map update of the last frame and the egress of its vectors; the flags that order the next frame
    // behind them stay as they are (they are satisfied now)
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (egress_stream_) CT_CUDA_CHECK(cudaStreamSynchronize(egress_stream_));
    const size_t T = trajectory_.size();
    const size_t map_size = map_->Save(nullptr, 0);
    const size_t total = OdoBlobSize(T, map_size);
    if (!dst || cap < total) return (int64_t) total;
    OdoHostRecord h{};
    h.registered_frames = registered_frames_;
    h.last_num_keypoints = (int64_t) last_num_keypoints_;
    h.next_robust_level = next_robust_level_;
    h.robust_num_consecutive_failures = robust_num_consecutive_failures_;
    h.suspect_registration_error = suspect_registration_error_ ? 1 : 0;
    h.tracker_skipped_frames = tracker_.skipped_frames;
    h.tracker_total_insertions = tracker_.total_insertions;
    h.tracker_cum_distance = tracker_.cum_distance;
    h.tracker_cum_orientation = tracker_.cum_orientation;
    h.default_motion_model_present = default_motion_model_.present ? 1 : 0;
    h.default_motion_model_options = default_motion_model_.options;
    h.default_motion_model_previous_frame = FrameToC(default_motion_model_.previous_frame);
    h.trajectory_size = T;
    std::vector<cticp_frame> tr(T);
    for (size_t i = 0; i < T; ++i) tr[i] = FrameToC(trajectory_[i]);
    OdoWrite(dst, options_, h, tr.data(), map_size);
    map_->Save(dst + OdoBlobSize(T, 0), map_size);
    SealBlob(dst, total);
    return (int64_t) total;
}

void Engine::LoadState(const uint8_t *src, size_t size) {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    if (shard_world_ > 1) throw UnsupportedError("load_state: restoring a sharded handle is not supported");
    const OdoBlobView v = OdoParse(src, size, true);
    const std::string diff = FirstOptionDifference(v.options, options_);
    if (!diff.empty()) throw std::invalid_argument("load_state: option " + diff + " differs from this handle's");
    const OdoHostRecord &h = v.host;
    if (h.next_robust_level < 0 || h.next_robust_level > options_.robust_minimal_level + 2)
        throw std::invalid_argument("state blob rejected: next_robust_level " + std::to_string(h.next_robust_level));
    std::vector<HostFrame> trajectory(h.trajectory_size);
    for (size_t i = 0; i < trajectory.size(); ++i) {
        cticp_frame f;
        memcpy(&f, v.trajectory + i, sizeof(f));
        trajectory[i] = FrameFromC(f);
    }
    // as Reset(): nothing in flight may still read or write the state that is replaced
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (egress_stream_) CT_CUDA_CHECK(cudaStreamSynchronize(egress_stream_));
    map_->Load(v.map, v.map_size);   // validates the map blob before it touches the map
    trajectory_ = std::move(trajectory);
    registered_frames_ = (int) h.registered_frames;
    last_num_keypoints_ = (size_t) h.last_num_keypoints;
    next_robust_level_ = h.next_robust_level;
    robust_num_consecutive_failures_ = h.robust_num_consecutive_failures;
    suspect_registration_error_ = h.suspect_registration_error != 0;
    tracker_.skipped_frames = h.tracker_skipped_frames;
    tracker_.total_insertions = h.tracker_total_insertions;
    tracker_.cum_distance = h.tracker_cum_distance;
    tracker_.cum_orientation = h.tracker_cum_orientation;
    default_motion_model_.present = h.default_motion_model_present != 0;
    default_motion_model_.options = h.default_motion_model_options;
    default_motion_model_.previous_frame = FrameFromC(h.default_motion_model_previous_frame);
    // the point vectors of the last registered frame are not state: get_points answers as on a new handle
    pipe_->ForgetFrame();
    last_frame_ = HostFrame();
    last_info_ = FrameInfo();
    frame_world_valid_ = last_all_world_valid_ = last_kp_world_valid_ = keypoints_in_summary_ = false;
    scan_in_staging_ = false;
    egress_pending_ = false;
    egress_valid_[0] = egress_valid_[1] = egress_valid_[2] = false;
    tail_event_valid_ = false;
    staging_in_flight_ = false;
    // LastTiming reads these once a frame was registered: recorded, they read as an empty interval
    for (int i = 0; i < 4; ++i) CT_CUDA_CHECK(cudaEventRecord(ev_[i], stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
}

void Engine::SetSummaryPoints(int mask) {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    summary_points_mask_ = mask & 7;
    if (summary_points_mask_) AllocEgress();
}
void Engine::AllocEgress() {
    if (!egress_stream_) {
        CT_CUDA_CHECK(cudaStreamCreateWithFlags(&egress_stream_, cudaStreamNonBlocking));
        CT_CUDA_CHECK(cudaEventCreateWithFlags(&ev_egress_main_, cudaEventDisableTiming));
        CT_CUDA_CHECK(cudaEventCreateWithFlags(&ev_egress_done_, cudaEventDisableTiming));
        for (auto &e : ev_egress_chunk_) CT_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const size_t cap = pipe_->MaxPoints();
    for (int i = 0; i < 3; ++i) {
        if (!(summary_points_mask_ & (1 << i))) continue;
        if (!h_world_[i]) CT_CUDA_CHECK(cudaMallocHost(&h_world_[i], sizeof(double) * 3 * cap));
        if (i != CTICP_POINTS_ALL_CORRECTED && !h_src_[i]) CT_CUDA_CHECK(cudaMallocHost(&h_src_[i], sizeof(uint32_t) * cap));
    }
    if (summary_points_mask_ & (1 << CTICP_POINTS_ALL_CORRECTED)) pipe_->EnsureAllWorld();
}

// World coordinates of the summary's three vectors → pinned host memory, on the egress stream: the transforms of all N
// points and of the keypoints run next to the map update of the main stream, the copies use the D2H engine. Called after
// the main stream has been synchronised on the pose read-back (so everything the egress kernels read is complete) and
// after TransformFrame was enqueued on the main stream (ev_egress_main_ orders the copy of d_frame_world behind it).
void Engine::EnqueueEgress(const HostFrame &f, bool ran_icp) {
    NvtxRange range("cticp.egress");
    const Q4 qb = f.begin_pose.pose.q, qe = f.end_pose.pose.q;
    const V3 tb = f.begin_pose.pose.t, te = f.end_pose.pose.t;
    const size_t n_all = pipe_->n(), n_frame = (size_t) pipe_->h_counts()[1];
    const size_t n_kp = (ran_icp && keypoints_in_summary_) ? (size_t) pipe_->h_counts()[2] : 0;
    cudaStream_t es = egress_stream_;
    if (summary_points_mask_ & (1 << CTICP_POINTS_ALL_CORRECTED)) {
        pipe_->TransformAll(qb, tb, qe, te, es);
        for (int c = 0; c < kEgressChunks; ++c) {
            const size_t b = n_all * (size_t) c / kEgressChunks, e = n_all * (size_t) (c + 1) / kEgressChunks;
            if (e > b)
                CT_CUDA_CHECK(cudaMemcpyAsync(h_world_[1] + 3 * b, pipe_->d_all_world() + 3 * b, sizeof(double) * 3 * (e - b),
                                              cudaMemcpyDeviceToHost, es));
            CT_CUDA_CHECK(cudaEventRecord(ev_egress_chunk_[c], es));
        }
        last_all_world_valid_ = true;
        egress_valid_[1] = true;
        egress_count_[1] = n_all;
        timing_.d2h_bytes += sizeof(double) * 3 * n_all;
    }
    if ((summary_points_mask_ & (1 << CTICP_POINTS_KEYPOINTS))) {
        if (n_kp) {
            pipe_->TransformInto(pipe_->d_keypoints(), pipe_->d_keypoints_lo(), pipe_->d_count_keypoints(), qb, tb, qe, te,
                                 d_kp_world_, es);
            CT_CUDA_CHECK(cudaMemcpyAsync(h_world_[2], d_kp_world_, sizeof(double) * 3 * n_kp, cudaMemcpyDeviceToHost, es));
            CT_CUDA_CHECK(cudaMemcpyAsync(h_src_[2], pipe_->d_keypoints_src(), sizeof(uint32_t) * n_kp, cudaMemcpyDeviceToHost, es));
            last_kp_world_valid_ = true;
        }
        egress_valid_[2] = true;
        egress_count_[2] = n_kp;
        timing_.d2h_bytes += (sizeof(double) * 3 + sizeof(uint32_t)) * n_kp;
    }
    if (summary_points_mask_ & (1 << CTICP_POINTS_CORRECTED)) {
        CT_CUDA_CHECK(cudaEventRecord(ev_egress_main_, stream_));          // d_frame_world is written by the main stream
        CT_CUDA_CHECK(cudaStreamWaitEvent(es, ev_egress_main_, 0));
        CT_CUDA_CHECK(cudaMemcpyAsync(h_world_[0], pipe_->d_frame_world(), sizeof(double) * 3 * n_frame, cudaMemcpyDeviceToHost, es));
        CT_CUDA_CHECK(cudaMemcpyAsync(h_src_[0], pipe_->d_frame_src(), sizeof(uint32_t) * n_frame, cudaMemcpyDeviceToHost, es));
        egress_valid_[0] = true;
        egress_count_[0] = n_frame;
        timing_.d2h_bytes += (sizeof(double) * 3 + sizeof(uint32_t)) * n_frame;
    }
    CT_CUDA_CHECK(cudaEventRecord(ev_egress_done_, es));
    egress_pending_ = true;
}

int64_t Engine::MapSize() {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    return (int64_t) map_->SyncCounters()[0].num_points;   // NumPoints(): resolution 0 only (map.h:345)
}

// InitializeMotion, odometry.cpp:276-330
void Engine::InitializeMotion(const FrameInfo &info, const cticp_frame *initial_estimate) {
    if (initial_estimate) {
        trajectory_.push_back(FrameFromC(*initial_estimate));
        return;
    }
    const int k = info.registered_fid;
    trajectory_.emplace_back();
    auto &T = trajectory_;
    T[k].begin_pose.dest_timestamp = info.begin_timestamp;
    T[k].begin_pose.dest_frame_id = info.frame_id;
    T[k].end_pose.dest_timestamp = info.end_timestamp;
    T[k].end_pose.dest_frame_id = info.frame_id;
    if (k <= 1) return;
    const bool cv = options_.initialization == CTICP_INIT_CONSTANT_VELOCITY;
    if (k == 2) {
        if (cv) {
            T[k].begin_pose.pose = T[k - 1].end_pose.pose;
            T[k].end_pose.pose = se3_mul(se3_mul(T[k - 1].end_pose.pose, se3_inverse(T[k - 2].end_pose.pose)), T[k - 1].end_pose.pose);
        } else {
            T[k].begin_pose.pose = T[k - 1].begin_pose.pose;
            T[k].end_pose.pose = T[k].begin_pose.pose;
        }
        return;
    }
    if (cv) {
        // CONTINUOUS: extrapolate the begin pose from the previous begin poses (:311-317); otherwise the new begin pose and
        // the previous end pose are made consistent (:318-321)
        if (options_.motion_compensation == CTICP_MC_CONTINUOUS)
            T[k].begin_pose.pose = se3_mul(se3_mul(T[k - 1].begin_pose.pose, se3_inverse(T[k - 2].begin_pose.pose)), T[k - 1].begin_pose.pose);
        else
            T[k].begin_pose.pose = T[k - 1].end_pose.pose;
        T[k].end_pose.pose = se3_mul(se3_mul(T[k - 1].end_pose.pose, se3_inverse(T[k - 2].end_pose.pose)), T[k - 1].end_pose.pose);
    } else {
        T[k].begin_pose.pose = T[k - 1].end_pose.pose;
        T[k].end_pose.pose = T[k - 1].end_pose.pose;
    }
}

// InitializeFrame, odometry.cpp:333-382 — host part: pack (x, y, z, alpha) into pinned memory; device part:
// shuffle / sub_sample_frame / timestamp override / shuffle.
void Engine::IngestImpl(const ScanView &scan, const FrameInfo &info, int64_t staged_slot) {
    NvtxRange range("cticp.ingest.subsample");
    const size_t n = scan.n;
    const int k = info.registered_fid;
    const HostFrame &tr = trajectory_[k];
    const double bts = tr.begin_pose.dest_timestamp, ets = tr.end_pose.dest_timestamp;
    // TPose::InterpolatePose CHECK (types.h:456): begin <= t <= end for every timestamp that gets interpolated
    const double t_lo = (k <= 1) ? info.end_timestamp : info.begin_timestamp, t_hi = info.end_timestamp;
    if (!(bts <= t_lo && t_hi <= ets)) {
        cudaStreamSynchronize(stream_);   // the scan's H2D copy may be in flight: leave the staging buffer quiescent
        staging_in_flight_ = false;
        throw TimestampError("The timestamp cannot be interpolated between the two poses");
    }
    if (n > pipe_->MaxPoints()) throw CapacityError("scan has more points than max_points_per_frame");

    // host buffers were packed and their H2D copy enqueued by PackAndUpload (RegisterCommon) before the pose pair existed
    if (staged_slot >= 0) pipe_->UploadFromDevice(staged_[staged_slot].d_points, staged_[staged_slot].d_lo, n);   // read in place
    timing_.h2d_bytes += pipe_->h2d_bytes();
    const double sample_size = k < options_.init_num_frames ? options_.init_voxel_size : options_.voxel_size;
    // frames 0 and 1: every timestamp := end_timestamp (odometry.cpp:355-359)
    const bool override_alpha = (k <= 1);
    const float alpha_value = (float) AlphaTimestamp(info.end_timestamp, bts, ets);
    // The keypoint sampling of the first registration attempt is known already (TryRegister: GRID sampling of the frame,
    // no truncation): both selections then run in ONE cooperative launch instead of six kernels and four memsets
    keypoints_sampled_ = false;
    const bool at_startup = k < options_.init_num_frames;
    // motion compensation CONSTANT_VELOCITY moves the raw points of the sub-sampled frame into the end pose's frame before
    // anything samples from it (DistortFrame, odometry.cpp:161-168,364-369)
    const bool distort = k > 1 && options_.motion_compensation == CTICP_MC_CONSTANT_VELOCITY;
    if (fused_sampling_ && !distort && k > 0 && !options_.robust_registration && options_.sampling == CTICP_SAMPLING_GRID &&
        (at_startup || options_.max_num_keypoints <= 0)) {
        const double kp_size = at_startup ? options_.init_sample_voxel_size : options_.sample_voxel_size;
        pipe_->SampleFused(sample_size, kp_size, options_.shuffle_seed, ShuffleCounter(k, 0), ShuffleCounter(k, 1),
                           override_alpha, alpha_value);
        keypoints_sampled_ = true;
        return;
    }
    pipe_->SubSampleFrame(sample_size, options_.shuffle_seed, ShuffleCounter(k, 0), ShuffleCounter(k, 1),
                          override_alpha, alpha_value);
    if (distort)
        pipe_->DistortFrame(tr.begin_pose.pose.q, tr.begin_pose.pose.t, tr.end_pose.pose.q, tr.end_pose.pose.t);
}

// Host team of the O(N) passes: half of the machine shared by the ranks of this node, 2..16 threads (measured on
// the 128-CPU B200 host: packing 130k points takes 0.25 ms on 2 threads, 0.085 on 8, 0.073 on 16).
int Engine::HostTeamSize(int ranks_on_node) {
    const int hw = std::max(1, (int) std::thread::hardware_concurrency());
    // half of the machine divided between the ranks (round 1 gave each rank hw / (4 ranks): 4 threads at 8 ranks on the
    // 128-CPU host, and the replicated packing — not the exchange — made the 8-GPU end-to-end time grow)
    int threads = std::max(2, std::min(16, hw / (2 * std::max(1, ranks_on_node))));
    if (ranks_on_node <= 1) threads = std::max(4, threads);
    if (const char *e = getenv("CTICP_HOST_THREADS")) threads = atoi(e);
    return std::max(1, std::min(threads, std::min(64, hw)));
}

// ---- host fork-join pool -------------------------------------------------------------------------------------
// The CPUs of the caller's socket (those the process may use): the team is kept on ONE socket. Measured on the 2 x 32-core
// host of the B200 box (profiles/README.md): a team scattered over both sockets packs a 130k-point scan in 145-175 us,
// the same team confined to either socket in 100-110 us (the pinned staging buffer and the caller's arrays are then
// local to everyone, and the parts' barrier does not cross the socket link).
static bool SocketCpuSet(cpu_set_t *out) {
    const char *env = getenv("CTICP_HOST_AFFINITY");
    if (env && atoi(env) == 0) return false;
    cpu_set_t allowed;
    if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return false;
    const int me = sched_getcpu();
    if (me < 0) return false;
    auto package_of = [](int cpu) {
        char path[128];
        snprintf(path, sizeof(path), "/sys/devices/system/cpu/cpu%d/topology/physical_package_id", cpu);
        FILE *f = fopen(path, "r");
        int id = -1;
        if (f) {
            if (fscanf(f, "%d", &id) != 1) id = -1;
            fclose(f);
        }
        return id;
    };
    const int mine = package_of(me);
    if (mine < 0) return false;
    CPU_ZERO(out);
    int count = 0, others = 0;
    for (int c = 0; c < CPU_SETSIZE; ++c) {
        if (!CPU_ISSET(c, &allowed)) continue;
        if (package_of(c) == mine) { CPU_SET(c, out); ++count; }
        else ++others;
    }
    return count >= 2 && others > 0;   // single-socket machines: nothing to do
}

HostPool::HostPool(int threads) {
    cpu_set_t socket;
    const bool pin = threads > 1 && SocketCpuSet(&socket);
    for (int i = 1; i < threads; ++i) {
        workers_.emplace_back([this, i] { Worker(i); });
        if (pin) pthread_setaffinity_np(workers_.back().native_handle(), sizeof(socket), &socket);   // best effort
    }
}
HostPool::~HostPool() {
    {
        std::lock_guard<std::mutex> lk(mu_);
        stop_ = true;
        generation_.fetch_add(1, std::memory_order_release);
    }
    cv_start_.notify_all();
    for (auto &w : workers_) w.join();
}
void HostPool::Worker(int id) {
    uint64_t seen = 0;
    while (true) {
        // poll for the next job for ~1 ms, then sleep. The first ~2k polls only pause (back-to-back frames find the
        // team awake); after that every poll also yields, so an oversubscribed host (several ranks per node, each
        // with its own team) is never held up by pollers
        bool have = false;
        const auto t0 = hclock::now();
        for (int spins = 0;; ++spins) {
            if (generation_.load(std::memory_order_acquire) != seen) {
                have = true;
                break;
            }
            _mm_pause();
            if (spins >= 2048) std::this_thread::yield();
            if ((spins & 255) == 255 && ms_since(t0) > 1.0) break;
        }
        if (!have) {
            std::unique_lock<std::mutex> lk(mu_);
            cv_start_.wait(lk, [&] { return generation_.load(std::memory_order_acquire) != seen; });
        }
        seen = generation_.load(std::memory_order_acquire);
        if (stop_) return;   // written before the generation bump that released us
        const std::function<void(int, int)> *fn = fn_;
        (*fn)(id, size());
        pending_.fetch_sub(1, std::memory_order_acq_rel);
    }
}
void HostPool::ParallelRegion(size_t n, const std::function<void(int, int)> &fn) {
    const int parts = PartsFor(n);
    if (parts == 1) {
        fn(0, 1);
        return;
    }
    {
        std::lock_guard<std::mutex> lk(mu_);   // orders the bump against a worker about to sleep on cv_start_
        fn_ = &fn;
        pending_.store(parts - 1, std::memory_order_relaxed);
        generation_.fetch_add(1, std::memory_order_release);
    }
    cv_start_.notify_all();
    fn(0, parts);
    for (int spins = 0; pending_.load(std::memory_order_acquire) != 0; ++spins) {
        if (spins < (1 << 16)) _mm_pause();
        else std::this_thread::yield();
    }
}
void HostPool::ParallelFor(size_t n, const std::function<void(size_t, size_t, int)> &fn) {
    ParallelRegion(n, [&](int part, int parts) {
        const size_t b = n * (size_t) part / (size_t) parts, e = n * (size_t) (part + 1) / (size_t) parts;
        if (e > b) fn(b, e, part);
    });
}

// (x, y, z, alpha) packing: alpha = GetAlphaTimestamp(t) w.r.t. the pose pair's timestamps (types.h:192-219);
// the caller has range-checked the timestamps
namespace {
template <typename T> struct TypeTag { using type = T; };
// calls fn(TypeTag<xyz scalar>, TypeTag<timestamp scalar>) for the view's dtypes
template <typename F> void DispatchScanTypes(const ScanView &v, F &&fn) {
    auto with_t = [&](auto xt) {
        switch (v.t_dtype) {
            case CTICP_DTYPE_INT8: fn(xt, TypeTag<int8_t>{}); break;
            case CTICP_DTYPE_UINT8: fn(xt, TypeTag<uint8_t>{}); break;
            case CTICP_DTYPE_INT16: fn(xt, TypeTag<int16_t>{}); break;
            case CTICP_DTYPE_UINT16: fn(xt, TypeTag<uint16_t>{}); break;
            case CTICP_DTYPE_INT32: fn(xt, TypeTag<int32_t>{}); break;
            case CTICP_DTYPE_UINT32: fn(xt, TypeTag<uint32_t>{}); break;
            case CTICP_DTYPE_FLOAT32: fn(xt, TypeTag<float>{}); break;
            case CTICP_DTYPE_FLOAT64: fn(xt, TypeTag<double>{}); break;
            default: throw std::invalid_argument("unknown timestamp dtype");
        }
    };
    switch (v.xyz_dtype) {
        case CTICP_DTYPE_FLOAT32: with_t(TypeTag<float>{}); break;
        case CTICP_DTYPE_FLOAT64: with_t(TypeTag<double>{}); break;
        default: throw std::invalid_argument("x/y/z must be FLOAT32 or FLOAT64");
    }
}
template <typename T> inline T LoadUnaligned(const char *p) {   // PointCloud2 records are packed: no alignment promise
    T v;
    memcpy(&v, p, sizeof(T));
    return v;
}
}  // namespace

namespace {
// one packed point: hi = float32(x, y, z, alpha) with a non-temporal store (the packed scan is consumed by the DMA engine,
// not by this core — keeping it out of the CPU caches took the H2D copy from ~12 GB/s, snooped dirty lines, to PCIe
// speed); for float64 sources also the residual plane lo = value - hi, and whether any coordinate needs it
template <typename XT>
inline void PackPoint(XT x, XT y, XT z, double a, float4 *dst, bool *any_lo) {
    const float fx = (float) x, fy = (float) y, fz = (float) z, fa = (float) a;
    _mm_stream_ps(reinterpret_cast<float *>(dst), _mm_set_ps(fa, fz, fy, fx));
    if constexpr (std::is_same<XT, double>::value) {
        // does any coordinate need the residual plane? (float64 arrays usually hold float32 values: then nothing more is
        // computed, stored or uploaded; otherwise PackLoPlane makes a second pass)
        if ((double) fx != x || (double) fy != y || (double) fz != z) *any_lo = true;
    }
}
// The common layout — contiguous float64 x, y, z and contiguous float64 timestamps (numpy's default) — has an AVX2 packer
// (host_pack.cpp: a plain C++ translation unit, nvcc's front end does not see the AVX intrinsics)
inline bool F64FastPath(const ScanView &scan) {
    static const bool avx2 = HostPackHasAvx2();
    return avx2 && scan.xyz_dtype == CTICP_DTYPE_FLOAT64 && scan.t_dtype == CTICP_DTYPE_FLOAT64 && scan.xyz_stride == 24 &&
           scan.t_stride == 8 && (reinterpret_cast<uintptr_t>(scan.xyz) & 7) == 0 && (reinterpret_cast<uintptr_t>(scan.t) & 7) == 0;
}
}  // namespace

// The residual plane of a float64 scan (value - (double)(float)value per component, alpha included): second pass, only for
// scans that need it.
void Engine::PackLoPlane(const ScanView &scan, double bts, double ets, float4 *dst_lo) {
    const double mn = std::min(bts, ets), mx = std::max(bts, ets);
    const bool spans = mx > mn;
    const double inv = spans ? 1.0 / (mx - mn) : 0.0;
    const char *px = static_cast<const char *>(scan.xyz), *pt = static_cast<const char *>(scan.t);
    const size_t xs = scan.xyz_stride, ts = scan.t_stride;
    DispatchScanTypes(scan, [&](auto xt, auto tt) {
        using XT = typename decltype(xt)::type;
        using TT = typename decltype(tt)::type;
        pool_->ParallelFor(scan.n, [&](size_t b, size_t e, int) {
            for (size_t i = b; i < e; ++i) {
                const char *p = px + i * xs;
                const double x = (double) LoadUnaligned<XT>(p), y = (double) LoadUnaligned<XT>(p + sizeof(XT)),
                             z = (double) LoadUnaligned<XT>(p + 2 * sizeof(XT));
                const double ti = (double) LoadUnaligned<TT>(pt + i * ts);
                const double a = spans ? (ti - mn) * inv : 1.0;
                _mm_stream_ps(reinterpret_cast<float *>(dst_lo + i),
                              _mm_set_ps((float) (a - (double) (float) a), (float) (z - (double) (float) z),
                                         (float) (y - (double) (float) y), (float) (x - (double) (float) x)));
            }
            _mm_sfence();
        });
    });
}

// returns whether the scan needs its residual plane (float64 coordinates that are not float32-representable)
bool Engine::PackScan(const ScanView &scan, double bts, double ets, float4 *dst) {
    std::atomic<bool> needs_lo{false};
    const double mn = std::min(bts, ets), mx = std::max(bts, ets);
    const double inv = (mx > mn) ? 1.0 / (mx - mn) : 0.0;
    const char *px = static_cast<const char *>(scan.xyz), *pt = static_cast<const char *>(scan.t);
    const size_t xs = scan.xyz_stride, ts = scan.t_stride;
    const bool spans = mx > mn;
    const bool fast = F64FastPath(scan);
    DispatchScanTypes(scan, [&](auto xt, auto tt) {
        using XT = typename decltype(xt)::type;
        using TT = typename decltype(tt)::type;
        pool_->ParallelFor(scan.n, [&](size_t b, size_t e, int) {
            bool any = false;
            if (fast) {   // slices cut on multiples of four points (the 32-byte stores need the alignment)
                const size_t bb = b & ~size_t(3), ee = e == scan.n ? e : e & ~size_t(3);
                if (ee > bb)
                    PackBlockF64Avx2(static_cast<const double *>(scan.xyz), static_cast<const double *>(scan.t), bb, ee, mn, inv,
                                     spans, dst, &any);
            }
            for (size_t i = b; i < e && !fast; ++i) {
                const char *p = px + i * xs;
                const XT x = LoadUnaligned<XT>(p), y = LoadUnaligned<XT>(p + sizeof(XT)), z = LoadUnaligned<XT>(p + 2 * sizeof(XT));
                const double ti = (double) LoadUnaligned<TT>(pt + i * ts);
                const double a = spans ? (ti - mn) * inv : 1.0;
                PackPoint<XT>(x, y, z, a, dst + i, &any);
            }
            _mm_sfence();
            if (any) needs_lo.store(true, std::memory_order_relaxed);
        });
    });
    return needs_lo.load();
}

// RegisterFrame's O(N) host work as ONE parallel region (one wake-up of the team instead of two):
//   1. every part reduces the timestamps of its slice to (min, max);
//   2. team barrier; the pose-pair timestamps are the scan's (min, max) (compute_frame_info, odometry.cpp:186-196)
//      unless the caller supplied an initial estimate (pose_timestamps = its {begin, end} dest_timestamp);
//   3. the scan is packed in kRounds rounds; in round r part p packs piece r * parts + p, so a finished round is one
//      contiguous range — part 0 enqueues its H2D copy at once and the copy engine works while later rounds are packed.
void Engine::PackAndUpload(const ScanView &scan, const double *pose_timestamps, double *mn_out, double *mx_out) {
    NvtxRange range("cticp.ingest.pack_upload");
    constexpr int kRounds = 4;
    const size_t n = scan.n;
    const int parts = pool_->PartsFor(n);
    const int rounds = parts == 1 ? 1 : kRounds;
    // with a team of four or more, part 0 (the caller's thread) packs nothing: it only enqueues the copy of each round the
    // moment the round is complete — its driver calls would otherwise sit on the packing's critical path
    const int first_packer = parts >= 4 ? 1 : 0, packers = parts - first_packer;
    const size_t pieces = (size_t) rounds * (size_t) packers;
    const char *px = static_cast<const char *>(scan.xyz), *pt = static_cast<const char *>(scan.t);
    const size_t xs = scan.xyz_stride, ts = scan.t_stride;
    float4 *dst = pipe_->Staging();
    std::atomic<bool> needs_lo{false};
    double mns[64], mxs[64];
    std::atomic<int> arrived{0};
    std::atomic<int> round_done[kRounds];
    for (auto &r : round_done) r.store(0, std::memory_order_relaxed);
    std::atomic<bool> failed{false};
    const bool debug = getenv("CTICP_DEBUG_TIMERS") != nullptr;
    // piece boundaries on multiples of 4 points (= one 64-byte line of the staging buffer per 4 NT stores)
    auto piece_begin = [&](size_t piece) { return piece >= pieces ? n : (n * piece / pieces) & ~size_t(3); };
    pipe_->UploadBegin(n);
    if (debug) cudaEventRecord(ev_[4], stream_);
    const bool fast = F64FastPath(scan);
    const auto t_region = hclock::now();
    double dbg_barrier_ms = 0, dbg_round_ms[kRounds] = {0, 0, 0, 0};   // part 0's view (CTICP_DEBUG_TIMERS)

    DispatchScanTypes(scan, [&](auto xt, auto tt) {
        using XT = typename decltype(xt)::type;
        using TT = typename decltype(tt)::type;
        pool_->ParallelRegion(n, [&](int part, int nparts) {
            // 1. min / max of my slice
            {
                const size_t b = n * (size_t) part / (size_t) nparts, e = n * (size_t) (part + 1) / (size_t) nparts;
                double mn = INFINITY, mx = -INFINITY;
                for (size_t i = b; i < e; ++i) {
                    const double ti = (double) LoadUnaligned<TT>(pt + i * ts);
                    mn = ti < mn ? ti : mn;
                    mx = ti > mx ? ti : mx;
                }
                mns[part] = mn;
                mxs[part] = mx;
            }
            // 2. team barrier (all parts are running: a short spin, yielding if the machine is oversubscribed)
            arrived.fetch_add(1, std::memory_order_acq_rel);
            for (int spins = 0; arrived.load(std::memory_order_acquire) < nparts; ++spins) {
                if (spins < 4096) _mm_pause();
                else std::this_thread::yield();
            }
            double smn = INFINITY, smx = -INFINITY;
            for (int i = 0; i < nparts; ++i) { smn = std::min(smn, mns[i]); smx = std::max(smx, mxs[i]); }
            if (part == 0) { *mn_out = smn; *mx_out = smx; }
            if (part == 0 && debug) dbg_barrier_ms = ms_since(t_region);
            const double bts = pose_timestamps ? pose_timestamps[0] : smn, ets = pose_timestamps ? pose_timestamps[1] : smx;
            const double mn = std::min(bts, ets), mx = std::max(bts, ets);
            const bool spans = mx > mn;
            const double inv = spans ? 1.0 / (mx - mn) : 0.0;
            // 3. packing in rounds; alpha = GetAlphaTimestamp(t) (types.h:192-219; the caller range-checks)
            int issued = 0;
            auto issue_ready = [&](bool wait_all) {   // part 0 only
                while (issued < rounds) {
                    if (round_done[issued].load(std::memory_order_acquire) < packers) {
                        if (!wait_all) return;
                        _mm_pause();
                        continue;
                    }
                    if (debug) dbg_round_ms[issued] = ms_since(t_region);
                    try {
                        pipe_->UploadRange(piece_begin((size_t) issued * packers), piece_begin((size_t) (issued + 1) * packers));
                    } catch (...) {
                        failed.store(true);
                    }
                    ++issued;
                }
            };
            bool any = false;
            for (int r = 0; r < rounds && part >= first_packer; ++r) {
                const size_t piece = (size_t) r * packers + (size_t) (part - first_packer);
                const size_t b = piece_begin(piece), e = piece_begin(piece + 1);
                if (fast && e > b)
                    PackBlockF64Avx2(static_cast<const double *>(scan.xyz), static_cast<const double *>(scan.t), b, e, mn, inv, spans,
                                     dst, &any);
                for (size_t i = b; i < e && !fast; ++i) {
                    const char *p = px + i * xs;
                    const XT x = LoadUnaligned<XT>(p), y = LoadUnaligned<XT>(p + sizeof(XT)), z = LoadUnaligned<XT>(p + 2 * sizeof(XT));
                    const double ti = (double) LoadUnaligned<TT>(pt + i * ts);
                    const double a = spans ? (ti - mn) * inv : 1.0;
                    PackPoint<XT>(x, y, z, a, dst + i, &any);
                }
                _mm_sfence();
                if (any) needs_lo.store(true, std::memory_order_relaxed);
                round_done[r].fetch_add(1, std::memory_order_acq_rel);
                if (part == 0) issue_ready(false);
            }
            if (part == 0) issue_ready(true);
        });
    });
    // float64 coordinates that float32 cannot hold: the residual plane follows (a second pass + one more copy; scans of
    // float32 values never get here)
    if (needs_lo.load()) {
        const double bts = pose_timestamps ? pose_timestamps[0] : *mn_out, ets = pose_timestamps ? pose_timestamps[1] : *mx_out;
        PackLoPlane(scan, bts, ets, pipe_->StagingLo());
        pipe_->UploadLo(n);
    }
    if (debug) {
        cudaEventRecord(ev_[5], stream_);
        fprintf(stderr, "[cticp] pack region (%d parts, %d packers): min/max + barrier at %.3f ms, rounds complete at %.3f %.3f %.3f %.3f, "
                "region end %.3f ms\n", parts, packers, dbg_barrier_ms, dbg_round_ms[0], dbg_round_ms[1], dbg_round_ms[2],
                dbg_round_ms[3], ms_since(t_region));
    }
    if (failed.load()) throw CudaError("cudaMemcpyAsync (scan upload)");
}

void Engine::MinMaxTimestamps(const ScanView &scan, double *mn_out, double *mx_out) {
    const char *pt = static_cast<const char *>(scan.t);
    const size_t ts = scan.t_stride;
    double mns[64], mxs[64];
    const int parts = pool_->size();
    for (int i = 0; i < parts; ++i) { mns[i] = INFINITY; mxs[i] = -INFINITY; }
    DispatchScanTypes(scan, [&](auto, auto tt) {
        using TT = typename decltype(tt)::type;
        pool_->ParallelFor(scan.n, [&](size_t b, size_t e, int part) {
            double mn = INFINITY, mx = -INFINITY;
            for (size_t i = b; i < e; ++i) {
                const double ti = (double) LoadUnaligned<TT>(pt + i * ts);
                mn = ti < mn ? ti : mn;
                mx = ti > mx ? ti : mx;
            }
            mns[part] = mn;
            mxs[part] = mx;
        });
    });
    double mn = INFINITY, mx = -INFINITY;
    for (int i = 0; i < parts; ++i) { mn = std::min(mn, mns[i]); mx = std::max(mx, mxs[i]); }
    *mn_out = mn;
    *mx_out = mx;
}

int64_t Engine::StageFrame(const ScanView &scan) {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    const size_t n = scan.n;
    if (n == 0 || !scan.xyz || !scan.t) throw std::invalid_argument("The registered frame cannot be empty");
    if (n > pipe_->MaxPoints()) throw CapacityError("scan has more points than max_points_per_frame");
    StagedScan sc;
    sc.n = n;
    MinMaxTimestamps(scan, &sc.t_min, &sc.t_max);
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));   // the pinned staging buffer may still feed a previous copy
    const bool needs_lo = PackScan(scan, sc.t_min, sc.t_max, pipe_->Staging());
    float4 *stage_lo = needs_lo ? pipe_->StagingLo() : nullptr;
    if (needs_lo) PackLoPlane(scan, sc.t_min, sc.t_max, stage_lo);
    CT_CUDA_CHECK(cudaMalloc(&sc.d_points, sizeof(float4) * n));
    CT_CUDA_CHECK(cudaMemcpyAsync(sc.d_points, pipe_->Staging(), sizeof(float4) * n, cudaMemcpyHostToDevice, stream_));
    if (needs_lo) {
        CT_CUDA_CHECK(cudaMalloc(&sc.d_lo, sizeof(float4) * n));
        CT_CUDA_CHECK(cudaMemcpyAsync(sc.d_lo, stage_lo, sizeof(float4) * n, cudaMemcpyHostToDevice, stream_));
    }
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    staged_.push_back(sc);
    return (int64_t) staged_.size() - 1;
}
void Engine::ClearStaged() {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    pipe_->DetachRaw();   // the last frame's points stay readable (GetPoints) after its staged scan is freed
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    for (auto &sc : staged_) { cudaFree(sc.d_points); cudaFree(sc.d_lo); }
    staged_.clear();
}
void Engine::TimerStart() {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    CT_CUDA_CHECK(cudaEventRecord(timer_ev_[0], stream_));
}
double Engine::TimerStop() {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    CT_CUDA_CHECK(cudaEventRecord(timer_ev_[1], stream_));
    CT_CUDA_CHECK(cudaEventSynchronize(timer_ev_[1]));
    float ms = 0.f;
    CT_CUDA_CHECK(cudaEventElapsedTime(&ms, timer_ev_[0], timer_ev_[1]));
    return (double) ms;
}
void Engine::FlushL2(size_t bytes) {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    if (bytes > flush_bytes_) {
        cudaFree(d_flush_);
        CT_CUDA_CHECK(cudaMalloc(&d_flush_, bytes));
        flush_bytes_ = bytes;
    }
    CT_CUDA_CHECK(cudaMemsetAsync(d_flush_, 0x5A, bytes, stream_));
}

// TryRegister, odometry.cpp:525-601
void Engine::TryRegister(const FrameInfo &info, cticp_icp_options &options, Summary &rs, double sample_voxel_size,
                         const MotionModel *mm, int attempt_idx) {
    NvtxRange range("cticp.icp");
    const int k = info.registered_fid;
    const bool at_startup = k < options_.init_num_frames;
    auto t0 = hclock::now();
    if (!(keypoints_sampled_ && attempt_idx == 0))   // (else: sampled together with the frame, IngestImpl)
        pipe_->SampleKeypoints(options_.sampling, sample_voxel_size,
                               (!at_startup && options_.max_num_keypoints > 0) ? options_.max_num_keypoints : -1,
                               options_.shuffle_seed, ShuffleCounter(k, 2 + attempt_idx), &options_.adaptive_options);
    keypoints_sampled_ = false;
    rs.t_sampling = ms_since(t0);
    if (callback_) {   // odometry.cpp:568: the keypoint count is needed on the host for the hook's GetPoints
        pipe_->QueueCountsReadback();
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        staging_in_flight_ = false;
        keypoints_in_summary_ = true;   // the hook receives the sampled keypoints (odometry.cpp:568)
        FireEvent(CTICP_EVENT_BEFORE_ITERATION, rs, info);
    }
    if (at_startup) {
        options.threshold_voxel_occupancy = 1;
        options.num_iters_icp = std::max(options.num_iters_icp, 15);
    }
    // registration state → device
    IcpState &S = *h_state_;
    memset(&S, 0, sizeof(S));
    const Q4 qb = qnormalized(rs.frame.begin_pose.pose.q), qe = qnormalized(rs.frame.end_pose.pose.q);
    S.qb[0] = qb.x; S.qb[1] = qb.y; S.qb[2] = qb.z; S.qb[3] = qb.w;
    S.qe[0] = qe.x; S.qe[1] = qe.y; S.qe[2] = qe.z; S.qe[3] = qe.w;
    const V3 tb = rs.frame.begin_pose.pose.t, te = rs.frame.end_pose.pose.t;
    S.tb[0] = tb.x; S.tb[1] = tb.y; S.tb[2] = tb.z;
    S.te[0] = te.x; S.te[1] = te.y; S.te[2] = te.z;
    if (mm && mm->present) {
        S.has_motion_model = 1;
        S.beta_location = mm->options.beta_location_consistency;
        S.beta_cv = mm->options.beta_constant_velocity;
        S.beta_small = mm->options.beta_small_velocity;
        S.beta_orientation = mm->options.beta_orientation_consistency;
        const auto &pf = mm->previous_frame;
        S.prev_tb[0] = pf.begin_pose.pose.t.x; S.prev_tb[1] = pf.begin_pose.pose.t.y; S.prev_tb[2] = pf.begin_pose.pose.t.z;
        S.prev_te[0] = pf.end_pose.pose.t.x; S.prev_te[1] = pf.end_pose.pose.t.y; S.prev_te[2] = pf.end_pose.pose.t.z;
        S.prev_qe[0] = pf.end_pose.pose.q.x; S.prev_qe[1] = pf.end_pose.pose.q.y; S.prev_qe[2] = pf.end_pose.pose.q.z;
        S.prev_qe[3] = pf.end_pose.pose.q.w;
    }
    icp_state_refresh_slerp(S);
    tail_launched_ = false;
    if (tail_armed_) {
        // nothing on stream_ touches d_state_ until the ICP kernel (the previous frame's readers completed before its verdict
        // arrived): the state goes up on the second stream while the sampler is still running
        CT_CUDA_CHECK(cudaMemcpyAsync(d_state_, h_state_, sizeof(IcpState), cudaMemcpyHostToDevice, aux_stream_));
        CT_CUDA_CHECK(cudaEventRecord(ev_state_up_, aux_stream_));
        CT_CUDA_CHECK(cudaStreamWaitEvent(stream_, ev_state_up_, 0));
    } else
        CT_CUDA_CHECK(cudaMemcpyAsync(d_state_, h_state_, sizeof(IcpState), cudaMemcpyHostToDevice, stream_));
    CT_CUDA_CHECK(cudaEventRecord(ev_[1], stream_));
    icp_->set_keypoints_lo(pipe_->d_keypoints_lo());
    FrameTailArgs tail{};
    bool verdict_by_icp_kernel = false;
    if (tail_armed_) {
        tail_in_.seq = ++verdict_seq_;
        tail.in = tail_in_;
        tail.counts = pipe_->d_counts();
        tail.dv = d_verdict_;
        tail.hv = h_verdict_dev_;
        tail.enabled = 1;
    }
    switch (options.solver) {
        case CTICP_SOLVER_GN:
            verdict_by_icp_kernel =
                icp_->EnqueueGaussNewton(*map_, options, pipe_->d_keypoints(), pipe_->d_count_keypoints(), KeypointHint(),
                                         options.num_iters_icp, d_state_, shard_rank_, shard_world_, nccl_comm_,
                                         (tail_armed_ && tail_in_kernel_) ? &tail : nullptr);
            break;
        case CTICP_SOLVER_CERES:
        case CTICP_SOLVER_ROBUST:
            icp_->EnqueueCeres(*map_, options, options_.neighborhood_strategy, pipe_->d_keypoints(),
                               pipe_->d_count_keypoints(), KeypointHint(), pipe_->n(), d_state_, shard_rank_, shard_world_,
                               nccl_comm_);
            break;
        default:
            throw UnsupportedError("Unsupported Solver Type");
    }
    CT_CUDA_CHECK(cudaEventRecord(ev_[2], stream_));
    if (tail_armed_) {
        // device tail (frame_policy.h): verdict + speculative map update behind the ICP kernel; the host waits for the
        // verdict's sequence number in mapped pinned memory, not for the stream
        tail_armed_ = false;
        if (!verdict_by_icp_kernel) {   // (k_gn_persistent's solver CTA writes the verdict itself)
            k_frame_policy<<<1, 32, 0, stream_>>>(d_state_, pipe_->d_counts(), tail_in_, d_verdict_, h_verdict_dev_);
            CT_CUDA_CHECK(cudaGetLastError());
            tail_launches_ += 1;
        }
        {
            NvtxRange range_map("cticp.map_update");
            map_->UpdateFused(pipe_->d_frame(), pipe_->d_frame_lo(), pipe_->d_count_frame(), pipe_->n(), pipe_->d_frame_world_mut(),
                              Q4{0, 0, 0, 1}, V3{0, 0, 0}, Q4{0, 0, 0, 1}, V3{0, 0, 0}, true, V3{0, 0, 0}, options_.max_distance,
                              true, V3{0, 0, 0}, d_verdict_);
        }
        tail_launched_ = true;
        WaitVerdict(tail_in_.seq);
        memcpy(h_state_, &h_verdict_->state, sizeof(IcpState));
        pipe_->SetHostCounts(h_verdict_->counts);
        timing_.d2h_bytes += sizeof(FrameVerdict);
    } else {
        CT_CUDA_CHECK(cudaMemcpyAsync(h_state_, d_state_, sizeof(IcpState), cudaMemcpyDeviceToHost, stream_));
        pipe_->QueueCountsReadback();
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        timing_.d2h_bytes += sizeof(IcpState) + sizeof(int) * 4;
    }
    staging_in_flight_ = false;
    icp_->CollectGatherTiming();
    timing_.h2d_bytes += sizeof(IcpState);

    if (getenv("CTICP_DEBUG_TIMERS"))
        fprintf(stderr, "[cticp] GN loop, solver CTA (SM cycles over %d iterations, needs a -DCTICP_DEBUG_TIMERS build): loop %llu, "
                "reduce+solve %llu = reduce %llu + rest %llu (12x12 solve %llu, pose update %llu)\n", (int) S.iter,
                (unsigned long long) S.cycles_total, (unsigned long long) S.cycles_solve, (unsigned long long) S.dbg_t[0],
                (unsigned long long) S.dbg_t[1], (unsigned long long) S.dbg_t[2], (unsigned long long) S.dbg_t[3]);
    if (getenv("CTICP_DEBUG_TIMERS") && options.solver == CTICP_SOLVER_GN) icp_->PrintWarpStamps((int) S.iter);
    rs.sample_size = pipe_->h_counts()[2];
    last_num_keypoints_ = (size_t) std::max(0, pipe_->h_counts()[2]);
    rs.icp.success = !S.failed;
    keypoints_in_summary_ = rs.icp.success;   // registration_summary.keypoints is only assigned after a successful ICP (odometry.cpp:584-597)
    rs.icp.num_residuals_used = S.n_used;
    rs.icp.num_iters = S.iter;
    rs.success = rs.icp.success;
    rs.number_of_residuals = S.n_used;
    timing_.icp_iterations += S.iter;
    timing_.gather_keypoint_iterations += S.stat_keypoint_iters;
    timing_.gather_stencil_points += S.stat_stencil_points;
    // the reference optimises frame_to_optimize in place, so even a failed ICP leaves its partial update behind
    rs.frame.begin_pose.pose.q = Q4{S.qb[0], S.qb[1], S.qb[2], S.qb[3]};
    rs.frame.end_pose.pose.q = Q4{S.qe[0], S.qe[1], S.qe[2], S.qe[3]};
    rs.frame.begin_pose.pose.t = V3{S.tb[0], S.tb[1], S.tb[2]};
    rs.frame.end_pose.pose.t = V3{S.te[0], S.te[1], S.te[2]};
    if (S.failed == 2) throw std::runtime_error("Error During Optimization");   // ct_icp.cpp:639-642
    if (S.failed == 3) throw std::runtime_error("multi-GPU exchange timed out: a peer rank never delivered its accumulator");
    if (S.failed == 4) {
        rs.error_message = "[CT_ICP]Error : the normal equations are singular (degenerate geometry and no regulariser)";
    } else if (!rs.success) {
        char buf[160];
        snprintf(buf, sizeof(buf), "[CT_ICP]Error : not enough keypoints selected in ct-icp ! Number_of_residuals : %d",
                 S.n_used);
        rs.error_message = buf;
    }
    // ICPSummary durations (ct_icp.cpp:664-666,690-694), milliseconds on the device: the ICP kernels between the two
    // events; the neighborhood / solve split of an iteration from the solver CTA's cycle stamps where the loop is one
    // persistent launch (solver GN), else the whole iteration is reported as neighborhood time
    {
        float icp_ms = 0.f;
        if (tail_launched_) cudaEventSynchronize(ev_[2]);   // (complete: the verdict's kernel ran behind it)
        if (cudaEventElapsedTime(&icp_ms, ev_[1], ev_[2]) != cudaSuccess) {
            cudaGetLastError();
            icp_ms = 0.f;
        }
        const int iters = std::max(1, (int) S.iter);
        rs.icp.duration_total = icp_ms;
        rs.icp.duration_init = 0.0;
        rs.icp.avg_duration_iter = icp_ms / iters;
        const double share = (S.cycles_total > 0) ? std::min(1.0, (double) S.cycles_solve / (double) S.cycles_total) : 0.0;
        rs.icp.avg_duration_solve = rs.icp.avg_duration_iter * share;
        rs.icp.avg_duration_neighborhood = rs.icp.avg_duration_iter - rs.icp.avg_duration_solve;
    }
    FireEvent(CTICP_EVENT_ITERATION_COMPLETED, rs, info);   // odometry.cpp:600
}

// Spin on the verdict's sequence number (written by k_frame_policy after a system-wide fence). The stream is polled now
// and then: a faulted kernel must surface as an error, not as a hang.
void Engine::WaitVerdict(unsigned seq) {
    volatile unsigned *flag = &h_verdict_->seq;
    for (unsigned long spins = 1;; ++spins) {
        if (*flag == seq) break;
        if ((spins & 0xfffu) == 0) {
            const cudaError_t q = cudaStreamQuery(stream_);
            if (q == cudaSuccess) {
                if (*flag == seq) break;
                throw std::runtime_error("the frame verdict never arrived although the stream is idle");
            }
            if (q != cudaErrorNotReady) CT_CUDA_CHECK(q);
        }
        _mm_pause();
    }
    std::atomic_thread_fence(std::memory_order_acquire);
}

// What UpdateMap (below) does on the host around its launch, for a map update the device has already decided and run.
void Engine::AdoptDeviceMapUpdate(Summary &s) {
    const FrameVerdict &v = *h_verdict_;
    const bool inserted = v.action == kFrameInsert;
    tracker_.cum_orientation += s.relative_orientation;
    tracker_.cum_distance += s.relative_distance;
    s.points_added = v.add_points_policy != 0;
    map_->CommitSpeculativeInsert(inserted);
    frame_world_valid_ = true;
    if (inserted) {
        tracker_.skipped_frames = 0;
        tracker_.cum_orientation = 0;
        tracker_.cum_distance = 0;
        tracker_.total_insertions++;
    } else
        tracker_.skipped_frames++;
    map_->QueueCounterReadback();
}

// AssessRegistration, odometry.cpp:604-684
bool Engine::AssessRegistration(Summary &s) const {
    if (s.relative_distance > options_.distance_error_threshold) return false;
    if (s.relative_orientation > options_.orientation_error_threshold ||
        s.ego_orientation > options_.orientation_error_threshold)
        return false;
    bool success = s.success;
    if (options_.robust_registration) {
        if (s.robust_level == 0 && (s.relative_orientation > options_.robust_threshold_relative_orientation ||
                                    s.ego_orientation > options_.robust_threshold_ego_orientation)) {
            if (s.robust_level < options_.robust_num_attempts_when_rotation) {
                s.error_message = "Large rotations require at a robust_level of at least 1 (got:" +
                                  std::to_string(s.robust_level) + ").";
                return false;
            }
        }
        if (s.relative_distance > options_.robust_relative_trans_threshold) {
            s.error_message = "The relative distance is too important";
            return false;
        }
    }
    return success;
}

// RobustRegistration + RobustRegistrationAttempt, odometry.cpp:780-852, 996-1050
void Engine::RobustRegistration(const FrameInfo &info, Summary &rs, const MotionModel *mm) {
    const int k = info.registered_fid;
    const HostFrame initial_estimate = rs.frame;
    cticp_icp_options reg = options_.ct_icp_options;
    int robust_level = 0;
    double sample_voxel_size = k < options_.init_num_frames ? options_.init_sample_voxel_size : options_.sample_voxel_size;
    Summary attempt = rs;
    attempt.number_of_attempts = 0;
    auto increase = [&]() {   // IncreaseRobustnessLevel, :996-1018
        const double min_voxel_size = std::min(options_.init_voxel_size, options_.voxel_size);
        attempt.frame = initial_estimate;
        reg.ls_max_num_iters += 30;
        if (reg.max_num_residuals > 0) reg.max_num_residuals = reg.max_num_residuals * 2;
        reg.num_iters_icp = std::min(reg.num_iters_icp + 20, 50);
        reg.threshold_orientation_norm = std::max(reg.threshold_orientation_norm / 10, 1.e-5);
        reg.threshold_translation_norm = std::max(reg.threshold_orientation_norm / 10, 1.e-4);
        sample_voxel_size = std::max(options_.sample_voxel_size / 1.5, double(min_voxel_size));
        reg.ls_sigma *= 1.2;
        reg.max_dist_to_plane_ct_icp *= 1.5;
        robust_level++;
    };
    while (robust_level < next_robust_level_) increase();
    bool good_enough = false;
    int attempt_idx = 0;
    do {
        TryRegister(info, reg, attempt, sample_voxel_size, mm, attempt_idx++);
        if (k > 0) {
            const auto &prev = trajectory_[k - 1];
            const V3 d = attempt.frame.begin_pose.pose.t - prev.end_pose.pose.t;
            attempt.distance_correction = norm(d);
            attempt.relative_orientation = angular_distance_deg(prev.end_pose.pose.q, attempt.frame.end_pose.pose.q);
            attempt.ego_orientation = EgoAngularDistance(attempt.frame);
        }
        attempt.relative_distance = norm(attempt.frame.end_pose.pose.t - attempt.frame.begin_pose.pose.t);
        good_enough = AssessRegistration(attempt);
        attempt.number_of_attempts++;
        if (!good_enough) {
            if (attempt.number_of_attempts < options_.robust_num_attempts)
                increase();
            else
                good_enough = true;
        }
    } while (!good_enough);
    rs = attempt;
    if (rs.number_of_attempts > options_.robust_num_attempts)
        robust_num_consecutive_failures_++;
    else
        robust_num_consecutive_failures_ = 0;
}

// ComputeSummaryMetrics, odometry.cpp:978-988
void Engine::ComputeSummaryMetrics(Summary &s, int k) {
    if (k > 0) {
        const auto &cur = trajectory_[k];
        const auto &prev = trajectory_[k - 1];
        s.distance_correction = norm(cur.begin_pose.pose.t - prev.end_pose.pose.t);
        s.relative_orientation = angular_distance_deg(prev.end_pose.pose.q, cur.end_pose.pose.q);
        s.relative_distance = norm(prev.end_pose.pose.t - cur.end_pose.pose.t);
        s.ego_orientation = EgoAngularDistance(cur);
    }
}

// UpdateMap, odometry.cpp:855-953
void Engine::UpdateMap(Summary &s, int registered_fid) {
    NvtxRange range("cticp.map_update");
    bool add_points = true;
    if (options_.robust_registration) {
        suspect_registration_error_ = s.number_of_attempts >= options_.robust_num_attempts;
        if (s.ego_orientation > options_.robust_threshold_ego_orientation ||
            s.relative_orientation > options_.robust_threshold_relative_orientation)
            add_points = false;
        if (suspect_registration_error_) add_points |= (robust_num_consecutive_failures_ > 5);
        next_robust_level_ = add_points ? options_.robust_minimal_level : options_.robust_minimal_level + 1;
        if (!s.success)
            next_robust_level_ = options_.robust_minimal_level + 2;
        else {
            if (s.relative_orientation > options_.robust_threshold_relative_orientation ||
                s.ego_orientation > options_.robust_threshold_ego_orientation)
                next_robust_level_ = options_.robust_minimal_level + 1;
            if (s.number_of_attempts > 1) next_robust_level_ = options_.robust_minimal_level + 1;
        }
    } else {
        tracker_.cum_orientation += s.relative_orientation;
        tracker_.cum_distance += s.relative_distance;
        if (tracker_.total_insertions > 0) {
            if (s.ego_orientation > options_.insertion_ego_rotation_threshold)
                add_points = tracker_.skipped_frames > options_.insertion_threshold_frames_skipped;
            else
                add_points = true;
        }
    }
    s.points_added = add_points;
    if (options_.do_no_insert) add_points = false;
    if (options_.always_insert) add_points = true;

    const V3 location = trajectory_.back().end_pose.pose.t;
    if (add_points) map_->EnsureRoomFor((size_t) std::max(0, pipe_->h_counts()[1]));   // F is known since the pose read-back
    if (fused_map_update_) {
        // transform of the sub-sampled frame + eviction + insertion on every resolution: one cooperative launch
        const auto &f = s.frame;
        map_->UpdateFused(pipe_->d_frame(), pipe_->d_frame_lo(), pipe_->d_count_frame(), pipe_->n(), pipe_->d_frame_world_mut(), f.begin_pose.pose.q,
                          f.begin_pose.pose.t, f.end_pose.pose.q, f.end_pose.pose.t, true, location, options_.max_distance,
                          add_points, f.begin_pose.pose.t);
        frame_world_valid_ = true;
    } else {
        map_->RemoveFar(location, options_.max_distance);
        // frame_poses = {begin_pose, end_pose} (odometry.cpp:949): the begin position orients the voxel normals
        if (add_points) map_->InsertDevice(pipe_->d_frame_world(), pipe_->d_count_frame(), pipe_->n(), s.frame.begin_pose.pose.t);
    }
    if (add_points) {
        tracker_.skipped_frames = 0;
        tracker_.cum_orientation = 0;
        tracker_.cum_distance = 0;
        tracker_.total_insertions++;
        (void) registered_fid;
    } else
        tracker_.skipped_frames++;
    map_->QueueCounterReadback();
}

// RegisterFrame / RegisterFrameWithEstimate (odometry.cpp:199-236) → DoRegister (:386-501)
void Engine::RegisterFrame(const ScanView &scan, uint32_t frame_id, const cticp_frame *initial_estimate,
                           cticp_summary *out, const cticp_motion_prior *motion_model) {
    if (scan.n == 0 || !scan.xyz || !scan.t) throw std::invalid_argument("The registered frame cannot be empty");
    RegisterCommon(scan, frame_id, initial_estimate, -1, out, motion_model);
}

// IterateOverCallbacks, odometry.cpp:742-750. The hook may fetch the frame / the keypoints (GetPoints) under the pose pair
// of this moment.
void Engine::FireEvent(int event, const Summary &rs, const FrameInfo &info) {
    if (!callback_) return;
    last_frame_ = rs.frame;
    last_info_ = info;
    frame_world_valid_ = last_all_world_valid_ = last_kp_world_valid_ = false;
    egress_valid_[0] = egress_valid_[1] = egress_valid_[2] = false;
    if (!callback_(event, callback_user_)) throw CallbackError("Callback returned false");
}
void Engine::RegisterStaged(int64_t slot, uint32_t frame_id, cticp_summary *out) {
    if (slot < 0 || slot >= (int64_t) staged_.size()) throw std::invalid_argument("unknown staged slot");
    ScanView none;
    none.n = staged_[slot].n;
    RegisterCommon(none, frame_id, nullptr, slot, out);
}

void Engine::RegisterCommon(const ScanView &scan, uint32_t frame_id, const cticp_frame *initial_estimate,
                            int64_t staged_slot, cticp_summary *out, const cticp_motion_prior *motion_model) {
    const size_t n = scan.n;
    auto t_start = hclock::now();
    CT_CUDA_CHECK(cudaSetDevice(device_));
    if (n > pipe_->MaxPoints()) throw CapacityError("scan has more points than max_points_per_frame");
    memset(&timing_, 0, sizeof(timing_));
    icp_->reset_timing();
    const int launches0 = map_->launches() + pipe_->launches() + icp_->launches() + tail_launches_;
    tail_armed_ = tail_launched_ = false;
    keypoints_in_summary_ = false;
    last_all_world_valid_ = last_kp_world_valid_ = frame_world_valid_ = false;
    egress_valid_[0] = egress_valid_[1] = egress_valid_[2] = false;
    if (egress_pending_) {   // the previous frame's egress still reads d_raw / d_frame_world / the keypoints
        CT_CUDA_CHECK(cudaStreamWaitEvent(stream_, ev_egress_done_, 0));
        egress_pending_ = false;
    }
    scan_in_staging_ = staged_slot < 0;

    // compute_frame_info, odometry.cpp:186-196
    FrameInfo info;
    double t_pack = 0;
    if (staged_slot >= 0) {
        info.begin_timestamp = staged_[staged_slot].t_min;
        info.end_timestamp = staged_[staged_slot].t_max;
    } else {
        // Host buffers: timestamp min/max, packing and the H2D copy, pipelined (PackAndUpload). The copy is enqueued
        // behind the previous frame's map update, which may still be running: the stream keeps the order, and the
        // pinned staging buffer is free (its previous copy completed before that frame's ICP state was read back).
        if (staging_in_flight_) CT_CUDA_CHECK(cudaStreamSynchronize(stream_));   // only after a call that threw midway
        staging_in_flight_ = true;
        CT_CUDA_CHECK(cudaEventRecord(ev_[0], stream_));
        double pose_ts[2];
        if (initial_estimate) {
            pose_ts[0] = initial_estimate->begin_pose.dest_timestamp;
            pose_ts[1] = initial_estimate->end_pose.dest_timestamp;
        }
        PackAndUpload(scan, initial_estimate ? pose_ts : nullptr, &info.begin_timestamp, &info.end_timestamp);
        t_pack = ms_since(t_start);
        if (getenv("CTICP_DEBUG_TIMERS")) fprintf(stderr, "[cticp] host min/max + pack + upload enqueue %.3f ms\n", t_pack);
    }
    info.registered_fid = registered_frames_++;
    info.frame_id = frame_id;
    const int k = info.registered_fid;
    InitializeMotion(info, initial_estimate);

    // the previous frame's map update: its counters tell whether the tables need maintenance. Waits on that frame's
    // last event, NOT on the stream — this frame's H2D copy is already in flight behind it.
    if (tail_event_valid_) CT_CUDA_CHECK(cudaEventSynchronize(ev_[3]));
    else CT_CUDA_CHECK(cudaStreamSynchronize(stream_));   // first frame, after Reset(), or after a call that threw
    tail_event_valid_ = false;
    map_->NotifyStreamSynchronized();
    map_->MaintainTables();

    if (staged_slot >= 0) CT_CUDA_CHECK(cudaEventRecord(ev_[0], stream_));
    IngestImpl(scan, info, staged_slot);
    const double t_initialization = ms_since(t_start);

    Summary summary;
    summary.frame = trajectory_.back();
    summary.initial_frame = summary.frame;
    bool early_return = false;
    bool ran_icp = false;
    if (k > 0) {
        const MotionModel *mm = nullptr;
        MotionModel caller_model;
        if (motion_model) {   // the caller's AMotionModel* (a PreviousFrameMotionModel in its current state)
            caller_model.present = true;
            caller_model.options = motion_model->options;
            caller_model.previous_frame = FrameFromC(motion_model->previous_frame);
            mm = &caller_model;
        } else if (options_.with_default_motion_model) {   // odometry.cpp:412-417
            default_motion_model_.present = true;
            default_motion_model_.options = options_.default_motion_model;
            default_motion_model_.previous_frame = trajectory_[k - 1];
            mm = &default_motion_model_;
        }
        ran_icp = true;
        if (options_.robust_registration) {
            RobustRegistration(info, summary, mm);
        } else {
            cticp_icp_options ct_icp_options = options_.ct_icp_options;
            const double sample_voxel_size = k < options_.init_num_frames ? options_.init_sample_voxel_size
                                                                          : options_.sample_voxel_size;
            auto t0 = hclock::now();
            // NB trajectory_[k] is still the INITIAL estimate here (odometry.cpp:429-431)
            const double relative_orientation =
                angular_distance_deg(trajectory_[k - 1].end_pose.pose.q, trajectory_[k].end_pose.pose.q);
            if (device_tail_ && fused_map_update_ && !callback_ && options_.motion_compensation == CTICP_MC_CONTINUOUS &&
                pipe_->n() > 0) {
                // the tail of this registration is decided on the device (frame_policy.h)
                FramePolicyIn &in = tail_in_;
                in = FramePolicyIn{};
                in.distance_error_threshold = options_.distance_error_threshold;
                in.orientation_error_threshold = options_.orientation_error_threshold;
                in.relative_orientation = relative_orientation;
                in.insertion_ego_rotation_threshold = options_.insertion_ego_rotation_threshold;
                in.quit_on_error = options_.quit_on_error ? 1 : 0;
                in.has_insertions = tracker_.total_insertions > 0;
                in.skipped_enough = tracker_.skipped_frames > options_.insertion_threshold_frames_skipped;
                in.do_no_insert = options_.do_no_insert ? 1 : 0;
                in.always_insert = options_.always_insert ? 1 : 0;
                // F is still on the device: room for the previous frame's count with head-room (a frame beyond it is
                // deferred to the host-side UpdateMap). Before the ICP is enqueued — a grown table is a new table.
                const size_t prev_f = (size_t) std::max(0, pipe_->h_counts()[1]);
                size_t room = std::min(pipe_->n(), prev_f + prev_f / 2 + 4096);
                if (const char *e = getenv("CTICP_TAIL_ROOM")) room = std::min(room, (size_t) std::max(0, atoi(e)));   // test hook: force the deferred path
                map_->EnsureRoomFor(room);
                in.room_for = (int) room;
                tail_armed_ = true;
            }
            TryRegister(info, ct_icp_options, summary, sample_voxel_size, mm, 0);
            summary.t_try_register = ms_since(t0);
            summary.relative_orientation = relative_orientation;
            summary.ego_orientation = EgoAngularDistance(summary.frame);
            summary.relative_distance = norm(summary.frame.end_pose.pose.t - summary.frame.begin_pose.pose.t);
            bool assessed = AssessRegistration(summary);
            if (tail_launched_) assessed = h_verdict_->assess_ok != 0;   // the device acted on ITS evaluation of the same formulas
            if (!assessed) {
                summary.success = false;
                if (options_.quit_on_error) early_return = true;
            }
        }
        if (!early_return) trajectory_[k] = summary.frame;
    } else {
        CT_CUDA_CHECK(cudaEventRecord(ev_[1], stream_));
        CT_CUDA_CHECK(cudaEventRecord(ev_[2], stream_));
        pipe_->QueueCountsReadback();
    }
    last_frame_ = summary.frame;
    last_info_ = info;

    auto t_before_map = hclock::now();
    if (!early_return) {
        const auto &f = summary.frame;
        if (!ran_icp) {   // frame 0: no pose read-back has synchronised the stream yet; F sizes the map tables / the egress
            pipe_->QueueCountsReadback();
            CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
            staging_in_flight_ = false;
        }
        if (!fused_map_update_) {
            pipe_->TransformFrame(f.begin_pose.pose.q, f.begin_pose.pose.t, f.end_pose.pose.q, f.end_pose.pose.t);
            frame_world_valid_ = true;
            if (summary_points_mask_) EnqueueEgress(f, ran_icp);
        }
        ComputeSummaryMetrics(summary, k);
        if (tail_launched_ && h_verdict_->action != kFrameDeferred)
            AdoptDeviceMapUpdate(summary);   // evicted / inserted already, behind the ICP kernel
        else
            UpdateMap(summary, k);
        if (fused_map_update_ && summary_points_mask_) EnqueueEgress(f, ran_icp);   // (the fused update wrote d_frame_world)
        if (callback_) {   // odometry.cpp:491
            const bool fw = frame_world_valid_, aw = last_all_world_valid_, kw = last_kp_world_valid_;
            const bool e0 = egress_valid_[0], e1 = egress_valid_[1], e2 = egress_valid_[2];
            FireEvent(CTICP_EVENT_FINISHED_REGISTRATION, summary, info);
            frame_world_valid_ = fw; last_all_world_valid_ = aw; last_kp_world_valid_ = kw;   // same pose pair: still valid
            egress_valid_[0] = e0; egress_valid_[1] = e1; egress_valid_[2] = e2;
        }
    }
    CT_CUDA_CHECK(cudaEventRecord(ev_[3], stream_));
    tail_event_valid_ = true;
    if (!ran_icp) {   // frame 0: counts for the summary
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        staging_in_flight_ = false;
    }

    timing_.kernel_launches = map_->launches() + pipe_->launches() + icp_->launches() + tail_launches_ - launches0;
    if (out) {
        FillSummary(summary, out);
        out->num_all_corrected_points = n;
        out->num_corrected_points = (uint64_t) pipe_->h_counts()[1];
        out->num_keypoints = (ran_icp && keypoints_in_summary_) ? (uint64_t) pipe_->h_counts()[2] : 0;
        out->odometry_total = ms_since(t_start);
        out->odometry_initialization = t_initialization;
        out->odometry_try_register = summary.t_try_register;
        out->odometry_duration_sampling = summary.t_sampling;
        out->odometry_map_update = ms_since(t_before_map);
        out->odometry_transform = 0;
    }
}

void Engine::FillSummary(const Summary &s, cticp_summary *out) const {
    memset(out, 0, sizeof(*out));
    out->frame = FrameToC(s.frame);
    out->initial_frame = FrameToC(s.initial_frame);
    out->icp_summary = s.icp;
    out->sample_size = s.sample_size;
    out->number_of_residuals = s.number_of_residuals;
    out->robust_level = s.robust_level;
    out->success = s.success;
    out->points_added = s.points_added;
    out->number_of_attempts = s.number_of_attempts;
    out->distance_correction = s.distance_correction;
    out->relative_distance = s.relative_distance;
    out->relative_orientation = s.relative_orientation;
    out->ego_orientation = s.ego_orientation;
    snprintf(out->error_message, sizeof(out->error_message), "%s", s.error_message.c_str());
}

cticp_device_timing Engine::LastTiming() {
    cudaSetDevice(device_);
    if (registered_frames_ == 0) {   // nothing recorded yet: querying the events would leave a sticky CUDA error
        cudaStreamSynchronize(stream_);
        return timing_;
    }
    cudaEventSynchronize(ev_[3]);
    float a = 0, b = 0, c = 0, d = 0;
    cudaEventElapsedTime(&a, ev_[0], ev_[1]);
    cudaEventElapsedTime(&b, ev_[1], ev_[2]);
    cudaEventElapsedTime(&c, ev_[2], ev_[3]);
    cudaEventElapsedTime(&d, ev_[0], ev_[3]);
    timing_.ingest_ms = a;
    timing_.icp_ms = b;
    timing_.map_update_ms = c;
    timing_.total_ms = d;
    timing_.gather_ms = icp_->gather_ms();
    timing_.gather_launches = icp_->gather_launches();
    if (getenv("CTICP_DEBUG_TIMERS")) {
        float h = 0, g = 0;
        if (cudaEventElapsedTime(&h, ev_[4], ev_[5]) == cudaSuccess && cudaEventElapsedTime(&g, ev_[0], ev_[4]) == cudaSuccess)
            fprintf(stderr, "[cticp] device: ev0->upload start %.3f ms, H2D %.3f ms\n", g, h);
        cudaGetLastError();
    }
    return timing_;
}

// RegistrationSummary::{corrected_points, all_corrected_points, keypoints} on demand
// the device arrays behind RegistrationSummary::{corrected_points, all_corrected_points, keypoints}
void Engine::ResolvePoints(int which, const float4 **out_pts, const float4 **out_lo, const double **out_world,
                           size_t *out_count) {
    CT_CUDA_CHECK(cudaSetDevice(device_));
    const float4 *d_pts = nullptr, *d_lo = nullptr;
    const double *d_world = nullptr;
    size_t count = 0;
    const auto &f = last_frame_;
    switch (which) {
        case CTICP_POINTS_CORRECTED:
            if (!frame_world_valid_) {
                pipe_->TransformFrame(f.begin_pose.pose.q, f.begin_pose.pose.t, f.end_pose.pose.q, f.end_pose.pose.t);
                frame_world_valid_ = true;
            }
            d_pts = pipe_->d_frame();
            d_lo = pipe_->d_frame_lo();
            d_world = pipe_->d_frame_world();
            count = (size_t) pipe_->h_counts()[1];
            break;
        case CTICP_POINTS_ALL_CORRECTED:
            if (!last_all_world_valid_) {
                pipe_->TransformAll(f.begin_pose.pose.q, f.begin_pose.pose.t, f.end_pose.pose.q, f.end_pose.pose.t);
                last_all_world_valid_ = true;
            }
            d_pts = pipe_->d_raw();
            d_lo = pipe_->d_raw_lo();
            d_world = pipe_->d_all_world();
            count = pipe_->n();
            break;
        case CTICP_POINTS_KEYPOINTS:
            count = (last_info_.registered_fid > 0 && keypoints_in_summary_) ? (size_t) pipe_->h_counts()[2] : 0;
            if (count && !last_kp_world_valid_) {
                pipe_->TransformInto(pipe_->d_keypoints(), pipe_->d_keypoints_lo(), pipe_->d_count_keypoints(), f.begin_pose.pose.q,
                                     f.begin_pose.pose.t, f.end_pose.pose.q, f.end_pose.pose.t, d_kp_world_);
                last_kp_world_valid_ = true;
            }
            d_pts = pipe_->d_keypoints();
            d_lo = pipe_->d_keypoints_lo();
            d_world = d_kp_world_;
            break;
        default:
            throw std::invalid_argument("which");
    }
    *out_pts = d_pts;
    *out_lo = d_lo;
    *out_world = d_world;
    *out_count = count;
}

int64_t Engine::GetPoints(int which, cticp_wpoint *dst, size_t cap) {
    // (a frame distorted on the device — motion compensation CONSTANT_VELOCITY — is no longer what the staging buffer holds)
    if (which >= 0 && which < 3 && egress_valid_[which] && scan_in_staging_ &&
        !(pipe_->frame_distorted() && which != CTICP_POINTS_ALL_CORRECTED)) {
        // eager path: the world coordinates (and source indices) are already on their way to pinned host memory; the raw
        // coordinates and the alpha timestamps are still in the pinned staging buffer the scan was packed into
        CT_CUDA_CHECK(cudaSetDevice(device_));
        const size_t count = egress_count_[which];
        const size_t m = std::min(cap, count);
        if (m == 0 || !dst) return (int64_t) count;
        const bool chunked = which == CTICP_POINTS_ALL_CORRECTED;   // copied first and in pieces (EnqueueEgress)
        if (!chunked) CT_CUDA_CHECK(cudaEventSynchronize(ev_egress_done_));
        const auto &f = last_frame_;
        const double bts = f.begin_pose.dest_timestamp, ets = f.end_pose.dest_timestamp;
        const double mn = std::min(bts, ets), mx = std::max(bts, ets);
        const float4 *stage = pipe_->Staging();
        const float4 *stage_lo = pipe_->StagingLoIfAny();
        const double *w = h_world_[which];
        const uint32_t *src = which == CTICP_POINTS_ALL_CORRECTED ? nullptr : h_src_[which];
        // frames 0 and 1: the sub-sampled frame (and its keypoints) carry timestamp := end_timestamp (odometry.cpp:355-359)
        const bool override_t = src && last_info_.registered_fid <= 1;
        const double t_override = mn + (double) (float) AlphaTimestamp(last_info_.end_timestamp, bts, ets) * (mx - mn);
        const uint32_t frame_id = last_info_.frame_id;
        const int pieces = chunked ? kEgressChunks : 1;
        for (int c = 0; c < pieces; ++c) {
        const size_t pb = chunked ? count * (size_t) c / kEgressChunks : 0;
        const size_t pe = std::min(m, chunked ? count * (size_t) (c + 1) / kEgressChunks : m);
        if (chunked) CT_CUDA_CHECK(cudaEventSynchronize(ev_egress_chunk_[c]));
        if (pe <= pb) continue;
        pool_->ParallelFor(pe - pb, [&](size_t b0, size_t e0, int) {
            for (size_t i = pb + b0; i < pb + e0; ++i) {
                const size_t si = src ? src[i] : i;
                const float4 p = stage[si];
                cticp_wpoint &o = dst[i];
                o.raw[0] = p.x; o.raw[1] = p.y; o.raw[2] = p.z;
                double alpha = (double) p.w;
                if (stage_lo) {
                    const float4 l = stage_lo[si];
                    o.raw[0] += (double) l.x; o.raw[1] += (double) l.y; o.raw[2] += (double) l.z;
                    alpha += (double) l.w;
                }
                o.timestamp = override_t ? t_override : mn + alpha * (mx - mn);
                o.world[0] = w[3 * i]; o.world[1] = w[3 * i + 1]; o.world[2] = w[3 * i + 2];
                o.index_frame = frame_id;
                o._pad0 = 0;
            }
        });
        }
        return (int64_t) count;
    }
    const float4 *d_pts = nullptr, *d_lo = nullptr;
    const double *d_world = nullptr;
    size_t count = 0;
    ResolvePoints(which, &d_pts, &d_lo, &d_world, &count);
    const auto &f = last_frame_;
    const size_t m = std::min(cap, count);
    if (m == 0 || !dst) return (int64_t) count;
    std::vector<float4> hp(m), hl(d_lo ? m : 0);
    std::vector<double> hw(3 * m);
    CT_CUDA_CHECK(cudaMemcpyAsync(hp.data(), d_pts, sizeof(float4) * m, cudaMemcpyDeviceToHost, stream_));
    if (d_lo) CT_CUDA_CHECK(cudaMemcpyAsync(hl.data(), d_lo, sizeof(float4) * m, cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaMemcpyAsync(hw.data(), d_world, sizeof(double) * 3 * m, cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    const double bts = f.begin_pose.dest_timestamp, ets = f.end_pose.dest_timestamp;
    const double mn = std::min(bts, ets), mx = std::max(bts, ets);
    for (size_t i = 0; i < m; ++i) {
        cticp_wpoint &o = dst[i];
        o.raw[0] = hp[i].x; o.raw[1] = hp[i].y; o.raw[2] = hp[i].z;
        double alpha = (double) hp[i].w;
        if (d_lo) {
            o.raw[0] += (double) hl[i].x; o.raw[1] += (double) hl[i].y; o.raw[2] += (double) hl[i].z;
            alpha += (double) hl[i].w;
        }
        o.timestamp = mn + alpha * (mx - mn);
        o.world[0] = hw[3 * i]; o.world[1] = hw[3 * i + 1]; o.world[2] = hw[3 * i + 2];
        o.index_frame = last_info_.frame_id;
        o._pad0 = 0;
    }
    return (int64_t) count;
}

// cticp_odometry_write_points: the same vectors written straight into the caller's record layout
int64_t Engine::WritePoints(int which, const cticp_cloud_sink &sink) {
    const float4 *d_pts = nullptr, *d_lo = nullptr;
    const double *d_world = nullptr;
    size_t count = 0;
    ResolvePoints(which, &d_pts, &d_lo, &d_world, &count);
    const size_t m = std::min((size_t) sink.capacity_points, count);
    if (m == 0 || !sink.data) return (int64_t) count;
    const size_t xs = sink.xyz_dtype == CTICP_DTYPE_FLOAT32 ? 4 : 8;
    if (sink.xyz_dtype != CTICP_DTYPE_FLOAT32 && sink.xyz_dtype != CTICP_DTYPE_FLOAT64)
        throw std::invalid_argument("sink: x/y/z must be FLOAT32 or FLOAT64");
    if (sink.t_dtype != 0 && sink.t_dtype != CTICP_DTYPE_FLOAT32 && sink.t_dtype != CTICP_DTYPE_FLOAT64)
        throw std::invalid_argument("sink: timestamp must be FLOAT32 or FLOAT64");
    if ((size_t) sink.xyz_offset + 3 * xs > sink.point_step ||
        (sink.t_dtype && (size_t) sink.t_offset + (sink.t_dtype == CTICP_DTYPE_FLOAT32 ? 4 : 8) > sink.point_step))
        throw std::invalid_argument("sink: a field lies outside the record (point_step)");
    std::vector<float4> hp(m), hl(d_lo ? m : 0);
    std::vector<double> hw(sink.world ? 3 * m : 0);
    CT_CUDA_CHECK(cudaMemcpyAsync(hp.data(), d_pts, sizeof(float4) * m, cudaMemcpyDeviceToHost, stream_));
    if (d_lo) CT_CUDA_CHECK(cudaMemcpyAsync(hl.data(), d_lo, sizeof(float4) * m, cudaMemcpyDeviceToHost, stream_));
    if (sink.world)
        CT_CUDA_CHECK(cudaMemcpyAsync(hw.data(), d_world, sizeof(double) * 3 * m, cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    const auto &f = last_frame_;
    const double bts = f.begin_pose.dest_timestamp, ets = f.end_pose.dest_timestamp;
    const double mn = std::min(bts, ets), mx = std::max(bts, ets);
    char *base = static_cast<char *>(sink.data);
    pool_->ParallelFor(m, [&](size_t b, size_t e, int) {
        for (size_t i = b; i < e; ++i) {
            char *rec = base + i * sink.point_step;
            double p[3];
            if (sink.world) { p[0] = hw[3 * i]; p[1] = hw[3 * i + 1]; p[2] = hw[3 * i + 2]; }
            else {
                p[0] = hp[i].x; p[1] = hp[i].y; p[2] = hp[i].z;
                if (d_lo) { p[0] += (double) hl[i].x; p[1] += (double) hl[i].y; p[2] += (double) hl[i].z; }
            }
            if (sink.xyz_dtype == CTICP_DTYPE_FLOAT32) {
                const float q[3] = {(float) p[0], (float) p[1], (float) p[2]};
                memcpy(rec + sink.xyz_offset, q, sizeof(q));
            } else {
                memcpy(rec + sink.xyz_offset, p, sizeof(p));
            }
            if (sink.t_dtype) {
                const double t = mn + ((double) hp[i].w + (d_lo ? (double) hl[i].w : 0.0)) * (mx - mn);
                if (sink.t_dtype == CTICP_DTYPE_FLOAT32) { const float tf = (float) t; memcpy(rec + sink.t_offset, &tf, 4); }
                else memcpy(rec + sink.t_offset, &t, 8);
            }
        }
    });
    return (int64_t) count;
}

}  // namespace cticp
