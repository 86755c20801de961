// device_map.h — host-side owner of the device-resident voxel map (see device_map.cuh for the layout).
#pragma once
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/cticp.h"
#include "device_map.cuh"

namespace cticp {

struct CudaError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct CapacityError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

struct FrameVerdict;   // frame_policy.h

class DeviceMap {
public:
    // with_normals: maintain the per-voxel normals that RadiusSearchInPlace's sensor_location filter reads (map.h:482-490)
    DeviceMap(const cticp_map_options &options, cudaStream_t stream, bool with_normals = false);
    ~DeviceMap();
    DeviceMap(const DeviceMap &) = delete;
    DeviceMap &operator=(const DeviceMap &) = delete;

    // InsertPointCloud (map.h:153-254): world points (fp64 xyz triples) already on the device, count on the device
    // `origin` = frame_poses.front().tr of the inserted frame (orients the normals, :222-226)
    void InsertDevice(const double *d_world_xyz, const int *d_n, size_t n_upper, V3 origin = V3{0, 0, 0});
    // same from strided host memory (synchronous; used by the cticp_map_* test entry points)
    void InsertHost(const double *xyz, size_t stride_bytes, size_t n, V3 origin = V3{0, 0, 0});
    bool HasNormals() const { return with_normals_; }
    // RemoveElementsFarFromLocation (map.h:305-322)
    void RemoveFar(V3 location, double distance);
    // one cooperative launch: world points of the sub-sampled frame under the pose pair (→ d_world), RemoveFar, InsertDevice
    void UpdateFused(const float4 *d_frame, const float4 *d_frame_lo, const int *d_n, size_t n_upper, double *d_world, const Q4 &qb, const V3 &tb,
                     const Q4 &qe, const V3 &te, bool do_remove, V3 location, double max_distance, bool do_insert, V3 origin,
                     const FrameVerdict *d_verdict = nullptr);
    // d_verdict != nullptr (frame_policy.h): a SPECULATIVE launch — the pose pair, the eviction centre and whether the frame
    // is evicted / inserted at all are read from the verdict on the device (the by-value pose arguments are ignored). The
    // caller reports the outcome it read back from the verdict:
    void CommitSpeculativeInsert(bool inserted) {
        if (inserted) ++frame_count_;
    }
    void Clear();

    // counters (synchronises the stream when stale)
    const MapCounters *SyncCounters();
    // enqueue the D2H of the counters; they are valid after the caller's next stream synchronisation
    void QueueCounterReadback();
    const MapCounters *HostCounters() const { return h_counters_; }
    void NotifyStreamSynchronized() { readback_pending_ = false; }
    void CheckOverflow();
    // tombstone purge / growth, driven by HostCounters(); call between frames
    void MaintainTables();
    // room for an insert of up to n_new points (grows / purges a table now if a probe sequence could wrap)
    void EnsureRoomFor(size_t n_new);

    // SearchParamsFromRadiusSearch (map.h:416-432)
    void SearchParams(double radius, int *level, int *voxel_neighborhood) const;
    const MapLevel &Level(int i) const { return levels_[i]; }
    int NumLevels() const { return (int) levels_.size(); }
    const cticp_map_options &Options() const { return options_; }
    cudaStream_t Stream() const { return stream_; }

    // GetMapPoints (map.h:354-376) in (voxel, insertion) order; returns the point count
    size_t Export(int level, std::vector<double> &xyz, std::vector<int> &voxels);
    // the map blob of state_io.h (canonical: voxels in ascending key order). Returns its size; writes only when
    // cap >= size. Synchronises the stream; the map itself is not changed.
    size_t Save(uint8_t *dst, size_t cap);
    // replaces the whole map by a validated blob of the same layout (levels, resolutions, normals); a rejected blob
    // (std::invalid_argument) leaves the map untouched
    void Load(const uint8_t *src, size_t size);

    int launches() const { return launches_; }
    int rebuilds() const { return rebuilds_; }

private:
    struct SortedLevel;
    // canonical order of the `num_voxels` live voxels (the level's counter; synchronises)
    std::unique_ptr<SortedLevel> SortLevel(int level, size_t num_voxels);
    uint64_t InitialCapacity(const cticp_resolution_param &rp) const;
    void AllocLevel(MapLevel &L, uint32_t cap, const cticp_resolution_param &rp);
    void RebuildLevel(size_t i, uint64_t new_cap);
    void FreeLevel(MapLevel &L);
    void EnsureScratch(size_t n_upper);
    void EnsureFrameOrigin();

    cticp_map_options options_;
    cudaStream_t stream_;
    std::vector<MapLevel> levels_;
    MapCounters *d_counters_ = nullptr;
    MapCounters *h_counters_ = nullptr;   // pinned
    void *d_scalar_ = nullptr;
    int *d_next_ = nullptr;
    uint32_t *d_touched_ = nullptr;
    size_t scratch_n_ = 0;
    double *d_world_tmp_ = nullptr;
    size_t world_tmp_n_ = 0;
    bool dirty_ = true;
    bool readback_pending_ = false;
    bool with_normals_ = false;
    double *d_frame_origins_ = nullptr;   // [3 * frame_capacity_] begin position of every inserted frame
    size_t frame_capacity_ = 0, frame_count_ = 0;
    int launches_ = 0;
    int rebuilds_ = 0;
    int fused_grid_ = 0;
};

}  // namespace cticp
