// engine.h — host orchestration of one odometry instance: the B200-native ct_icp::Odometry.
//
// Mirrors the control flow of src/ct_icp/odometry.cpp (RegisterFrame :199-214, InitializeMotion :276-330,
// InitializeFrame :333-382, DoRegister :386-501, TryRegister :525-601, AssessRegistration :604-684,
// RobustRegistration :780-852, UpdateMap :855-953) while every O(N)/O(K·S) stage runs on the device.
#pragma once
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/cticp.h"
#include "device_map.h"
#include "frame_pipeline.h"
#include "icp.h"
#include "frame_policy.h"

namespace cticp {

struct UnsupportedError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct TimestampError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

struct HostPose {   // slam::TPose<double>
    Se3 pose = se3_identity();
    double ref_timestamp = 0, dest_timestamp = -1;
    uint32_t ref_frame_id = 0, dest_frame_id = uint32_t(-1);
};
struct HostFrame {   // ct_icp::TrajectoryFrame
    HostPose begin_pose, end_pose;
};

// A borrowed scan: x,y,z contiguous of one scalar type at `xyz`, one timestamp scalar at `t`, both strided in bytes.
// What the reference reads through XYZConst<double>() / TimestampsProxy<double>() (odometry.cpp:335-336): any source
// scalar type, converted with static_cast<double> by the proxy (include/SlamCore/data/view.h:99-120).
struct ScanView {
    const void *xyz = nullptr;
    size_t xyz_stride = 0;
    int xyz_dtype = CTICP_DTYPE_FLOAT64;   // FLOAT32 / FLOAT64
    const void *t = nullptr;
    size_t t_stride = 0;
    int t_dtype = CTICP_DTYPE_FLOAT64;     // any CTICP_DTYPE_*
    size_t n = 0;
};

// host_pack.cpp: (x, y, z, alpha) packing of points [b, e) of a contiguous float64 scan with AVX2; b a multiple of 4.
// *any_lo is set when some coordinate is not float32-representable (never cleared).
bool HostPackHasAvx2();
void PackBlockF64Avx2(const double *xyz, const double *t, size_t b, size_t e, double mn, double inv, bool spans, float4 *dst,
                      bool *any_lo);

// Minimal fork-join pool for the host passes over a scan (timestamp min/max, float4 packing): the only O(N) host
// work of RegisterFrame. After a job the workers keep polling for the next one for ~1 ms before they go to sleep on a
// condition variable (what OpenMP runtimes do by default, cf. GOMP_SPINCOUNT): when frames arrive back to back the
// team starts within a microsecond instead of a futex wake-up per worker (~50 us for 15 workers); at sensor rate
// (10-20 Hz) the polling is a ~1 % duty cycle. The caller polls for completion as well (the job is ~50 us long).
struct CallbackError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

class HostPool {
public:
    explicit HostPool(int threads);
    ~HostPool();
    int size() const { return (int) workers_.size() + 1; }
    // number of parts a pass over n items is split into (1 below the threading threshold)
    int PartsFor(size_t n) const { return (size() == 1 || n < 16384) ? 1 : size(); }
    // fn(part, parts) on every thread of the team at once (parts = PartsFor(n)); the caller runs part 0. All parts run
    // concurrently, so fn may synchronise its parts (TeamBarrier)
    void ParallelRegion(size_t n, const std::function<void(int, int)> &fn);
    // fn(begin, end, part) over [0, n) split into PartsFor(n) contiguous parts
    void ParallelFor(size_t n, const std::function<void(size_t, size_t, int)> &fn);

private:
    void Worker(int id);
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_start_;
    const std::function<void(int, int)> *fn_ = nullptr;
    std::atomic<uint64_t> generation_{0};
    std::atomic<int> pending_{0};
    bool stop_ = false;
};

class Engine {
public:
    Engine(const cticp_odometry_options &options, int device);
    ~Engine();

    void RegisterFrame(const ScanView &scan, uint32_t frame_id, const cticp_frame *initial_estimate, cticp_summary *out,
                       const cticp_motion_prior *motion_model = nullptr);
    void SetCallback(cticp_event_fn fn, void *user) { callback_ = fn; callback_user_ = user; }
    const cticp_odometry_options &Options() const { return options_; }
    // device-resident input: pack + copy a scan to HBM now, register it later
    int64_t StageFrame(const ScanView &scan);
    int64_t WritePoints(int which, const cticp_cloud_sink &sink);
    void RegisterStaged(int64_t slot, uint32_t frame_id, cticp_summary *out);
    void ClearStaged();
    void TimerStart();
    double TimerStop();
    void FlushL2(size_t bytes);
    int64_t GetPoints(int which, cticp_wpoint *dst, size_t cap);
    // RegistrationSummary's point vectors (odometry.cpp:462-486,597) produced EAGERLY by every RegisterFrame: bit
    // `which` of the mask (CTICP_POINTS_*) selects a vector. 0 (default): computed on demand by GetPoints / WritePoints.
    void SetSummaryPoints(int mask);
    const std::vector<HostFrame> &Trajectory() const { return trajectory_; }
    int64_t MapSize();
    void Reset();
    // checkpoint / resume (state_io.h): everything that influences the frames to come. SaveState returns the blob size
    // and writes only when cap >= size; it waits for the work in flight and leaves the handle as it was. LoadState
    // replaces the whole state (also of a handle that registered frames already); a rejected blob changes nothing.
    int64_t SaveState(uint8_t *dst, size_t cap);
    void LoadState(const uint8_t *src, size_t size);
    DeviceMap &Map() { return *map_; }
    IcpSolver &Solver() { return *icp_; }
    cudaStream_t Stream() const { return stream_; }
    int Device() const { return device_; }
    cticp_device_timing LastTiming();   // synchronises on the last frame's final event
    void SetTimeGather(bool on) { icp_->set_time_gather(on); }
    void EnableSharding(const void *unique_id, int rank, int world);
    void DestroySharding();
    int ShardingMode() const { return shard_world_ <= 1 ? 0 : (icp_ && icp_->peers_ready() ? 2 : 1); }

private:
    struct FrameInfo {
        int registered_fid = -1;
        uint32_t frame_id = uint32_t(-1);
        double begin_timestamp = -1, end_timestamp = -1;
    };
    struct Summary {   // RegistrationSummary minus the point vectors
        HostFrame frame, initial_frame;
        int sample_size = 0, number_of_residuals = 0, robust_level = 0;
        double distance_correction = 0, relative_distance = 0, relative_orientation = 0, ego_orientation = 0;
        bool success = true, points_added = false;
        int number_of_attempts = 0;
        std::string error_message;
        cticp_icp_summary icp{};
        double t_try_register = 0, t_sampling = 0;
    };
    struct MotionModel {
        bool present = false;
        cticp_motion_model_options options{};
        HostFrame previous_frame;
    };

    void InitializeMotion(const FrameInfo &info, const cticp_frame *initial_estimate);
    void ResolvePoints(int which, const float4 **out_pts, const float4 **out_lo, const double **out_world, size_t *out_count);
    void IngestImpl(const ScanView &scan,
                    const FrameInfo &info, int64_t staged_slot);
    bool PackScan(const ScanView &scan, double bts, double ets, float4 *dst);
    void PackLoPlane(const ScanView &scan, double bts, double ets, float4 *dst_lo);
    // one parallel region: timestamp min/max → team barrier → (x, y, z, alpha) packing in rounds, the H2D copy of a
    // round enqueued as soon as the round is complete (the copy engine runs while the later rounds are still packed)
    void PackAndUpload(const ScanView &scan, const double *pose_timestamps, double *mn_out, double *mx_out);
    void MinMaxTimestamps(const ScanView &scan, double *mn_out, double *mx_out);
    std::unique_ptr<HostPool> pool_;
    static int HostTeamSize(int ranks_on_node);
    void RegisterCommon(const ScanView &scan, uint32_t frame_id, const cticp_frame *initial_estimate,
                        int64_t staged_slot, cticp_summary *out, const cticp_motion_prior *motion_model = nullptr);
    void FireEvent(int event, const Summary &rs, const FrameInfo &info);
    cticp_event_fn callback_ = nullptr;
    void *callback_user_ = nullptr;
    bool frame_world_valid_ = false;
    bool fused_map_update_ = true;     // CTICP_FUSED_MAP_UPDATE=0: transform / evict / insert as separate launches
    bool fused_sampling_ = true;       // CTICP_FUSED_SAMPLING=0: the two grid selections as separate launches
    bool keypoints_sampled_ = false;   // the keypoints of the coming first attempt were sampled with the frame   // d_frame_world holds the sub-sampled frame under last_frame_
    struct StagedScan {
        float4 *d_points = nullptr;
        float4 *d_lo = nullptr;   // residual plane, float64 scans only (se3.cuh load_raw)
        size_t n = 0;
        double t_min = 0, t_max = 0;
    };
    std::vector<StagedScan> staged_;
    cudaEvent_t timer_ev_[2];
    void *d_flush_ = nullptr;
    size_t flush_bytes_ = 0;
    void TryRegister(const FrameInfo &info, cticp_icp_options &options, Summary &rs, double sample_voxel_size,
                     const MotionModel *mm, int attempt_idx);
    bool AssessRegistration(Summary &s) const;
    void RobustRegistration(const FrameInfo &info, Summary &rs, const MotionModel *mm);
    void ComputeSummaryMetrics(Summary &s, int k);
    void UpdateMap(Summary &s, int registered_fid);
    // The tail of a plain registration decided on the device (frame_policy.h): TryRegister enqueues k_frame_policy and a
    // speculative k_map_update_fused right behind the ICP kernel, then waits for the verdict in mapped pinned memory — no
    // copy-engine operation and no host round trip between the ICP loop and the map update.
    bool device_tail_ = true;      // CTICP_DEVICE_TAIL=0: AssessRegistration / UpdateMap on the host for every frame
    bool tail_in_kernel_ = false;  // CTICP_TAIL_IN_KERNEL=1: solver GN's persistent kernel decides the tail itself at the end of
                                   // its loop instead of a separate k_frame_policy launch (three launches per frame; measured
                                   // neutral, profiles/r03h_bench*.json: 0.2479 vs 0.2483 ms per step — the default keeps the
                                   // policy in its own one-warp kernel, the same for every solver)
    bool tail_armed_ = false;      // the coming TryRegister enqueues the device tail (tail_in_ is filled)
    bool tail_launched_ = false;   // the last TryRegister did: h_verdict_ holds this frame's verdict
    FramePolicyIn tail_in_{};
    FrameVerdict *d_verdict_ = nullptr;
    FrameVerdict *h_verdict_ = nullptr;       // mapped pinned memory
    FrameVerdict *h_verdict_dev_ = nullptr;   // its device address
    unsigned verdict_seq_ = 0;
    int tail_launches_ = 0;
    void WaitVerdict(unsigned seq);
    void AdoptDeviceMapUpdate(Summary &s);
    // the registration state goes up on a second stream while the sampler runs (the ICP kernel waits for its event)
    cudaStream_t aux_stream_ = nullptr;
    cudaEvent_t ev_state_up_ = nullptr;
    void FillSummary(const Summary &s, cticp_summary *out) const;
    // grid-size hint for the ICP kernels: the keypoint count is only known on the device when they are enqueued, so
    // the host sizes the grid from the previous registration (keypoint counts change slowly) with 25% head-room;
    // the kernels stay correct for any count (warps loop)
    size_t KeypointHint() const {
        return last_num_keypoints_ ? std::min(pipe_->n(), last_num_keypoints_ + last_num_keypoints_ / 4 + 64) : pipe_->n();
    }
    size_t last_num_keypoints_ = 0;
    bool keypoints_in_summary_ = false;   // the last TryRegister's ICP succeeded: RegistrationSummary::keypoints is filled
    static uint64_t ShuffleCounter(int registered_fid, int purpose) {
        return (uint64_t(uint32_t(registered_fid)) << 8) | uint64_t(purpose & 0xff);
    }

    cticp_odometry_options options_;
    int device_;
    cudaStream_t stream_ = nullptr;
    std::unique_ptr<DeviceMap> map_;
    std::unique_ptr<FramePipeline> pipe_;
    std::unique_ptr<IcpSolver> icp_;
    IcpState *d_state_ = nullptr;
    IcpState *h_state_ = nullptr;   // pinned
    std::vector<HostFrame> trajectory_;
    MotionModel default_motion_model_;
    int registered_frames_ = 0;
    int robust_num_consecutive_failures_ = 0;
    bool suspect_registration_error_ = false;
    int next_robust_level_ = 0;
    struct {
        double cum_distance = 0, cum_orientation = 0;
        int skipped_frames = 0, total_insertions = 0;
    } tracker_;
    // state of the last registered frame (for GetPoints)
    HostFrame last_frame_;
    FrameInfo last_info_;
    bool last_all_world_valid_ = false, last_kp_world_valid_ = false;
    double *d_kp_world_ = nullptr;
    // eager egress of the summary vectors: world coordinates (+ source indices) to pinned host memory on a second
    // stream, overlapped with the map update; GetPoints assembles the 64-byte records on the host team
    void EnqueueEgress(const HostFrame &f, bool ran_icp);
    void AllocEgress();
    int summary_points_mask_ = 0;
    cudaStream_t egress_stream_ = nullptr;
    cudaEvent_t ev_egress_main_ = nullptr, ev_egress_done_ = nullptr;
    static constexpr int kEgressChunks = 4;            // the N world points go back in pieces: the host assembles the
    cudaEvent_t ev_egress_chunk_[kEgressChunks] = {};  // records of piece i while piece i + 1 is still on the bus
    bool egress_pending_ = false;           // ev_egress_done_ recorded, next frame's upload must wait for it
    bool egress_valid_[3] = {false, false, false};
    size_t egress_count_[3] = {0, 0, 0};
    double *h_world_[3] = {nullptr, nullptr, nullptr};   // pinned: corrected / all corrected / keypoints, xyz triples
    uint32_t *h_src_[3] = {nullptr, nullptr, nullptr};   // pinned: index into the scan (corrected, keypoints)
    bool scan_in_staging_ = false;          // the pinned staging buffer holds the last registered scan
    // timing
    cticp_device_timing timing_{};
    cudaEvent_t ev_[6];
    bool tail_event_valid_ = false;    // ev_[3] (end of the last frame's map update) has been recorded and not yet waited on
    bool staging_in_flight_ = false;   // the pinned staging buffer may still feed an H2D copy
    // multi-GPU
    void *nccl_comm_ = nullptr;
    int shard_rank_ = 0, shard_world_ = 1;
    // NVLink peer mailboxes of the in-kernel exchange (peer_exchange.cuh, nccl_shard.cu)
    bool ConnectPeers();
    void DisconnectPeers();
    void *d_mailbox_ = nullptr;
    std::vector<void *> peer_mapped_;
};

// conversions shared with capi.cu
HostPose PoseFromC(const cticp_pose &c);
cticp_pose PoseToC(const HostPose &p);
HostFrame FrameFromC(const cticp_frame &c);
cticp_frame FrameToC(const HostFrame &f);

}  // namespace cticp
