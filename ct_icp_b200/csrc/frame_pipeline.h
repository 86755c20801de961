// frame_pipeline.h — device buffers and kernels of one scan's journey: pinned staging → raw float4 → sub-sampled
// frame → keypoints → world-space frame (for the map). See frame_pipeline.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "device_map.h"
#include "se3.cuh"

namespace cticp {

class FramePipeline {
public:
    FramePipeline(size_t max_points, cudaStream_t stream);
    ~FramePipeline();
    FramePipeline(const FramePipeline &) = delete;
    FramePipeline &operator=(const FramePipeline &) = delete;

    // pinned staging buffer the host packs (x, y, z, alpha) into, then Upload(n) enqueues the H2D copy
    float4 *Staging() { return h_stage_; }
    // residual planes (value - (double)(float)value, see load_raw in se3.cuh) — allocated on first use: float32 scans,
    // what LiDAR drivers emit, never need them. raw_lo: the scan as uploaded; frame_lo: the sub-sampled frame and the
    // keypoints drawn from it (also set by DistortFrame, whose output is not float32-representable).
    void EnsureLo();
    float4 *StagingLo() { EnsureLo(); return h_stage_lo_; }
    const float4 *StagingLoIfAny() const { return raw_lo_ ? h_stage_lo_ : nullptr; }
    void UploadLo(size_t n);                                  // after Upload*/UploadBegin of the same scan
    bool raw_has_lo() const { return raw_lo_; }
    bool frame_has_lo() const { return frame_lo_; }
    bool frame_distorted() const { return distorted_; }
    const float4 *d_raw_lo() const { return raw_lo_ ? raw_lo_view_ : nullptr; }
    const float4 *d_frame_lo() const { return frame_lo_ ? d_frame_lo_ : nullptr; }
    const float4 *d_keypoints_lo() const { return frame_lo_ ? d_kp_lo_ : nullptr; }
    size_t MaxPoints() const { return max_points_; }
    void Upload(size_t n);
    // the same copy in pieces, so that it can start while the tail of the scan is still being packed:
    // UploadBegin(n), then UploadRange over a partition of [0, n) in any order
    void UploadBegin(size_t n);
    void UploadRange(size_t begin, size_t end);
    // a scan already packed and resident in HBM: the pipeline reads it where it is (no copy) until the next Upload* or
    // DetachRaw; N reaches the device with the sampler's launch
    void UploadFromDevice(const float4 *d_src, const float4 *d_src_lo, size_t n);
    // copy a resident scan the pipeline reads in place into its own buffers (before that scan's memory is freed)
    void DetachRaw();

    // Odometry::InitializeFrame: shuffle → sub_sample_frame → (frames 0,1: timestamp := end) → shuffle
    void SubSampleFrame(double voxel_size, uint64_t seed, uint64_t counter1, uint64_t counter2, bool override_alpha,
                        float alpha_value);
    // both of the above (GRID sampling, no truncation) in one cooperative launch
    void SampleFused(double voxel_size, double sample_voxel_size, uint64_t seed, uint64_t counter1, uint64_t counter2,
                     bool override_alpha, float alpha_value);
    // TryRegister: grid_sampling | NONE, then the optional max_num_keypoints shuffle-truncate
    void SampleKeypoints(int sampling, double sample_voxel_size, int max_num_keypoints, uint64_t seed, uint64_t counter,
                         const cticp_adaptive_options *adaptive = nullptr);
    // AdaptiveSamplePointsInGrid (include/ct_icp/algorithm/sampling.h:55-110)
    void AdaptiveSelect(const cticp_adaptive_options &o, const float4 *in, const float4 *in_lo, const uint32_t *in_src,
                        const int *d_n_in, size_t n_upper, float4 *out, float4 *out_lo, uint32_t *out_src, int *d_n_out);
    // DistortFrame (odometry.cpp:161-168) on the sub-sampled frame, in place
    void DistortFrame(const Q4 &qb, const V3 &tb, const Q4 &qe, const V3 &te);
    // world points of the sub-sampled frame / of every input point with the final pose pair
    void TransformFrame(const Q4 &qb, const V3 &tb, const Q4 &qe, const V3 &te);
    // (stream: nullptr = the pipeline's own; the egress of the summary vectors runs on a second stream)
    void TransformAll(const Q4 &qb, const V3 &tb, const Q4 &qe, const V3 &te, cudaStream_t stream = nullptr);
    void TransformInto(const float4 *pts, const float4 *lo, const int *d_n, const Q4 &qb, const V3 &tb, const Q4 &qe,
                       const V3 &te, double *d_world, cudaStream_t stream = nullptr);
    void EnsureAllWorld();

    void QueueCountsReadback();   // h_counts()[0..2] = N, F, K after the next stream sync
    const int *h_counts() const { return h_counts_; }
    // the same four counters, brought back by another route (the frame verdict, frame_policy.h)
    void SetHostCounts(const int *c) {
        for (int i = 0; i < 4; ++i) h_counts_[i] = c[i];
    }
    const int *d_counts() const { return d_counts_; }
    // no frame registered yet, as on a new pipeline (N and the host counters zero)
    void ForgetFrame() {
        n_ = 0;
        for (int i = 0; i < 4; ++i) h_counts_[i] = 0;
    }

    const float4 *d_raw() const { return raw_; }
    const float4 *d_frame() const { return d_frame_; }
    const float4 *d_keypoints() const { return d_keypoints_; }
    float4 *d_keypoints_mut() { return d_keypoints_; }
    const uint32_t *d_frame_src() const { return d_frame_src_; }
    const uint32_t *d_keypoints_src() const { return d_kp_src_; }
    const double *d_frame_world() const { return d_frame_world_; }
    const double *d_all_world() const { return d_all_world_; }
    int *d_count_n() { return d_counts_ + 0; }
    int *d_count_frame() { return d_counts_ + 1; }
    int *d_count_keypoints() { return d_counts_ + 2; }
    size_t n() const { return n_; }
    size_t h2d_bytes() const { return h2d_bytes_; }
    int launches() const { return launches_; }

    // generic "first-seen per voxel" selection (also behind cticp_grid_sample_indices)
    void GridSelect(const float4 *in, const float4 *in_lo, const uint32_t *in_src, const int *d_n_in, size_t n_upper,
                    double voxel_size, int use_perm1, uint64_t seed, uint64_t c1, int use_perm2, uint64_t c2,
                    int override_alpha, float alpha_value, float4 *out, float4 *out_lo, uint32_t *out_src, int *d_n_out);
    float4 *d_frame_lo_mut() { EnsureLo(); return d_frame_lo_; }
    double *d_frame_world_mut() { return d_frame_world_; }
    float4 *d_frame_mut() { return d_frame_; }
    uint32_t *d_frame_src_mut() { return d_frame_src_; }

private:
    int Blocks(size_t n) const;
    void EnsureCountN();   // counts[0] = N on the device, unless the sampler already wrote it

    cudaStream_t stream_;
    size_t max_points_, n_ = 0, h2d_bytes_ = 0;
    uint32_t grid_cap_ = 0;
    float4 *h_stage_ = nullptr;
    int *h_counts_ = nullptr;
    float4 *d_raw_ = nullptr, *d_frame_ = nullptr, *d_keypoints_ = nullptr, *d_tmp_points_ = nullptr;
    float4 *h_stage_lo_ = nullptr, *d_raw_lo_ = nullptr, *d_frame_lo_ = nullptr, *d_kp_lo_ = nullptr, *d_tmp_lo_ = nullptr;
    bool raw_lo_ = false, frame_lo_ = false, distorted_ = false;
    const float4 *raw_ = nullptr, *raw_lo_view_ = nullptr;   // the scan's planes: d_raw_ / d_raw_lo_ or a resident scan
    bool count_n_pending_ = false;
    uint32_t *d_frame_src_ = nullptr, *d_kp_src_ = nullptr, *d_tmp_src_ = nullptr;
    unsigned long long *d_grid_ = nullptr, *d_grid2_ = nullptr;
    int *d_slot_of_ = nullptr;
    uint32_t *d_tile_count_ = nullptr, *d_flags_ = nullptr, *d_src_ = nullptr;   // flags live right after the tile counters
    int *d_counts_ = nullptr;
    double *d_frame_world_ = nullptr, *d_all_world_ = nullptr;
    uint32_t *d_tile2_ = nullptr, *d_src2_ = nullptr;   // second selection of the fused sampler
    int fused_grid_ = 0;
    // k_sample_fused leaves the hash grid and selection 1's flag / tile arrays clean for the next frame (CTICP_SAMPLE_PRECLEAR=0:
    // every launch clears them itself): the capacity / word count that are clean right now
    bool preclear_ = true;
    uint32_t clean_cap_ = 0;
    size_t clean_words_ = 0;
    uint32_t *d_adaptive_ = nullptr;   // tile counters + flags + src of the band-major position space
    size_t adaptive_capacity_ = 0;
    int launches_ = 0;
};

}  // namespace cticp
