// state_io.h — the byte layout of saved odometry / map state (DESIGN.md §9). The only module that knows it: DeviceMap
// and Engine hand it counts and buffers and receive offsets, so neither reads or writes a header field itself.
//
// Map blob (little-endian, every section 8-byte aligned):
//   0  char[8] "CTICPMAP"   8  u32 version (1)   12 u32 num_levels   16 u64 total_bytes   24 u64 checksum
//   32 u32 has_normals       36 u32 0             40 u64 frame_count
//   48 f64 frame_origins[3 * frame_count]                     (has_normals only)
//   per level: f64 resolution, f64 min_distance_between_points, i32 max_num_points, i32 0, u64 V, u64 P,
//              u64 keys[V] (strictly ascending packed voxel keys), u32 counts[V] (zero-padded to 8 bytes),
//              float4 points[P] (stored bits: offset from the voxel origin, w = +-(frame ordinal + 1); the runs of the
//              voxels in key order, insertion order inside a run), f64 normals[4 * V] (has_normals only)
// Odometry blob:
//   0  char[8] "CTICPODO"   8  u32 version (1)   12 u32 sizeof(cticp_odometry_options)   16 u64 total_bytes
//   24 u64 checksum   32 cticp_odometry_options (effective options, padding zeroed)   then OdoHostRecord,
//   then cticp_frame trajectory[T], then one complete map blob up to total_bytes.
// checksum: FNV-1a 64 over bytes [32, total_bytes) taken as little-endian u64 words (h ^= word; h *= prime), the last
// word zero-padded. It detects truncation and corruption, not tampering: the loader validates the content as well.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/cticp.h"

namespace cticp {

constexpr uint32_t kStateVersion = 1;
constexpr size_t kMapHeaderBytes = 48;
constexpr size_t kOdoHeaderBytes = 32;
constexpr size_t kMapLevelHeaderBytes = 40;

uint64_t StateChecksum(const uint8_t *blob, size_t total);

// ---- map blob ----
struct MapBlobLevel {
    double resolution = 0, min_distance = 0;
    int max_num_points = 0;
    uint64_t V = 0, P = 0;
    size_t off_keys = 0, off_counts = 0, off_points = 0, off_normals = 0;   // byte offsets from the blob's start
};
struct MapBlobLayout {
    int num_levels = 0;
    bool has_normals = false;
    uint64_t frame_count = 0;
    size_t off_origins = 0;
    MapBlobLevel levels[CTICP_MAX_RESOLUTIONS];
    size_t total = 0;
};
// offsets of a blob holding levels[i].V voxels / levels[i].P points (the other fields of `L` are inputs too)
void MapLayoutFill(MapBlobLayout &L);
// header + per-level headers; the caller fills the sections, then SealBlob
void MapWriteHeaders(uint8_t *dst, const MapBlobLayout &L);
void SealBlob(uint8_t *blob, size_t total);
// every check of DESIGN.md §9 (magic, version, size, checksum, keys strictly ascending and inside +-2^20, counts <= B,
// P == sum of counts, point ordinals within frame_count, frame_count < 2^24 - 2); throws std::invalid_argument
MapBlobLayout MapParse(const uint8_t *src, size_t size);

// ---- odometry blob ----
struct OdoHostRecord {   // Engine's cross-frame host state (Engine::Reset lists it)
    int64_t registered_frames;
    int64_t last_num_keypoints;   // grid-size hint of the ICP kernels: fixes their summation order
    int32_t next_robust_level, robust_num_consecutive_failures;
    int32_t suspect_registration_error, tracker_skipped_frames;
    int32_t tracker_total_insertions, default_motion_model_present;
    double tracker_cum_distance, tracker_cum_orientation;
    cticp_motion_model_options default_motion_model_options;
    cticp_frame default_motion_model_previous_frame;
    uint64_t trajectory_size;
};
static_assert(sizeof(OdoHostRecord) % 8 == 0, "sections stay 8-byte aligned");

// the options as stored: padding fields zeroed
cticp_odometry_options CanonicalOptions(const cticp_odometry_options &o);
// name of the first field in which a and b differ, "" when equal; capacity_voxels / max_points_per_frame only size
// device buffers and are not compared
std::string FirstOptionDifference(const cticp_odometry_options &a, const cticp_odometry_options &b);

struct OdoBlobView {
    cticp_odometry_options options;
    OdoHostRecord host;
    const cticp_frame *trajectory;   // unaligned view into the blob: copy with memcpy
    const uint8_t *map;
    size_t map_size;
};
size_t OdoBlobSize(size_t trajectory_size, size_t map_size);
// writes header, options, host record and trajectory; the map blob goes to dst + OdoBlobSize(T, 0); then SealBlob
void OdoWrite(uint8_t *dst, const cticp_odometry_options &options, const OdoHostRecord &host, const cticp_frame *trajectory,
              size_t map_size);
// header, version, option size, total size and checksum (throws std::invalid_argument); full=true also splits off the
// trajectory and the map blob (which MapParse then validates)
OdoBlobView OdoParse(const uint8_t *src, size_t size, bool full);

}  // namespace cticp
