// state_io.cu — layout, checksum and validation of saved state (see state_io.h; DESIGN.md §9). Host code only.
#include "state_io.h"

#include <cmath>
#include <cstring>
#include <stdexcept>

#include "device_map.cuh"

namespace cticp {

namespace {
const char kMapMagic[8] = {'C', 'T', 'I', 'C', 'P', 'M', 'A', 'P'};
const char kOdoMagic[8] = {'C', 'T', 'I', 'C', 'P', 'O', 'D', 'O'};

size_t Align8(size_t v) { return (v + 7) & ~size_t(7); }
template <typename T>
T Get(const uint8_t *p) {
    T v;
    memcpy(&v, p, sizeof(T));
    return v;
}
template <typename T>
void Put(uint8_t *p, T v) {
    memcpy(p, &v, sizeof(T));
}
[[noreturn]] void Bad(const std::string &what) { throw std::invalid_argument("state blob rejected: " + what); }

// header common to both blobs: magic, version, total_bytes == size, checksum
void CheckHeader(const uint8_t *src, size_t size, const char *magic, const char *kind) {
    if (!src) Bad("null buffer");
    if (size < 32) Bad(std::string(kind) + " truncated (" + std::to_string(size) + " bytes)");
    if (memcmp(src, magic, 8) != 0) Bad(std::string("bad magic, expected ") + kind);
    if (Get<uint32_t>(src + 8) != kStateVersion)
        Bad(std::string(kind) + " version " + std::to_string(Get<uint32_t>(src + 8)) + " (this build reads " +
            std::to_string(kStateVersion) + ")");
    const uint64_t total = Get<uint64_t>(src + 16);
    if (total != size) Bad(std::string(kind) + " holds " + std::to_string(size) + " bytes, its header says " + std::to_string(total));
    if (total % 8) Bad(std::string(kind) + " size is not a multiple of 8");
    if (Get<uint64_t>(src + 24) != StateChecksum(src, size)) Bad(std::string(kind) + " checksum mismatch");
}
}  // namespace

uint64_t StateChecksum(const uint8_t *blob, size_t total) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (size_t o = 32; o < total; o += 8) {
        uint64_t w = 0;
        memcpy(&w, blob + o, std::min<size_t>(8, total - o));
        h ^= w;
        h *= 0x100000001b3ull;
    }
    return h;
}

void SealBlob(uint8_t *blob, size_t total) { Put<uint64_t>(blob + 24, StateChecksum(blob, total)); }

void MapLayoutFill(MapBlobLayout &L) {
    size_t o = kMapHeaderBytes;
    L.off_origins = o;
    if (L.has_normals) o += 24 * L.frame_count;
    for (int l = 0; l < L.num_levels; ++l) {
        MapBlobLevel &v = L.levels[l];
        o += kMapLevelHeaderBytes;
        v.off_keys = o;
        o += 8 * v.V;
        v.off_counts = o;
        o += Align8(4 * v.V);
        v.off_points = o;
        o += 16 * v.P;
        v.off_normals = o;
        if (L.has_normals) o += 32 * v.V;
    }
    L.total = o;
}

void MapWriteHeaders(uint8_t *dst, const MapBlobLayout &L) {
    memset(dst, 0, kMapHeaderBytes);
    memcpy(dst, kMapMagic, 8);
    Put<uint32_t>(dst + 8, kStateVersion);
    Put<uint32_t>(dst + 12, (uint32_t) L.num_levels);
    Put<uint64_t>(dst + 16, (uint64_t) L.total);
    Put<uint32_t>(dst + 32, L.has_normals ? 1u : 0u);
    Put<uint64_t>(dst + 40, L.frame_count);
    for (int l = 0; l < L.num_levels; ++l) {
        const MapBlobLevel &v = L.levels[l];
        uint8_t *h = dst + v.off_keys - kMapLevelHeaderBytes;
        memset(h, 0, kMapLevelHeaderBytes);
        Put<double>(h, v.resolution);
        Put<double>(h + 8, v.min_distance);
        Put<int32_t>(h + 16, v.max_num_points);
        Put<uint64_t>(h + 24, v.V);
        Put<uint64_t>(h + 32, v.P);
        if (v.V % 2) Put<uint32_t>(dst + v.off_counts + 4 * v.V, 0u);   // padding of the counts
    }
}

MapBlobLayout MapParse(const uint8_t *src, size_t size) {
    CheckHeader(src, size, kMapMagic, "map blob");
    if (size < kMapHeaderBytes) Bad("map blob truncated");
    MapBlobLayout L;
    const uint32_t levels = Get<uint32_t>(src + 12);
    if (levels < 1 || levels > CTICP_MAX_RESOLUTIONS) Bad("num_levels " + std::to_string(levels));
    L.num_levels = (int) levels;
    const uint32_t hn = Get<uint32_t>(src + 32);
    if (hn > 1 || Get<uint32_t>(src + 36) != 0) Bad("has_normals field");
    L.has_normals = hn == 1;
    L.frame_count = Get<uint64_t>(src + 40);
    if (L.frame_count >= (1u << 24) - 2) Bad("frame_count " + std::to_string(L.frame_count) + " >= 2^24 - 2");
    // walk the level headers with bounds checks before any section is read
    size_t o = kMapHeaderBytes + (L.has_normals ? 24 * L.frame_count : 0);
    for (int l = 0; l < L.num_levels; ++l) {
        if (o + kMapLevelHeaderBytes > size) Bad("map blob truncated in level " + std::to_string(l));
        MapBlobLevel &v = L.levels[l];
        v.resolution = Get<double>(src + o);
        v.min_distance = Get<double>(src + o + 8);
        v.max_num_points = Get<int32_t>(src + o + 16);
        v.V = Get<uint64_t>(src + o + 24);
        v.P = Get<uint64_t>(src + o + 32);
        if (Get<int32_t>(src + o + 20) != 0) Bad("level header padding");
        const uint64_t room = (uint64_t) size;   // every voxel takes >= 12 bytes and every point 16: bounds V and P
        if (v.V > room / 12 || v.P > room / 16) Bad("level " + std::to_string(l) + " sizes exceed the blob");
        o += kMapLevelHeaderBytes + 8 * v.V + Align8(4 * v.V) + 16 * v.P + (L.has_normals ? 32 * v.V : 0);
        if (o > size) Bad("map blob truncated in level " + std::to_string(l));
    }
    MapLayoutFill(L);
    if (L.total != size) Bad("map blob size " + std::to_string(size) + " != layout size " + std::to_string(L.total));
    const int64_t lim = kVoxelBias;
    for (int l = 0; l < L.num_levels; ++l) {
        const MapBlobLevel &v = L.levels[l];
        const std::string lv = "level " + std::to_string(l) + ": ";
        if (!(v.resolution > 0) || v.max_num_points < 1) Bad(lv + "resolution / max_num_points");
        unsigned long long prev = 0;
        uint64_t sum = 0;
        for (uint64_t i = 0; i < v.V; ++i) {
            const unsigned long long k = Get<uint64_t>(src + v.off_keys + 8 * i);
            if (k == kEmptyKey || k == kTombKey) Bad(lv + "sentinel key at voxel " + std::to_string(i));
            if (k >> 63) Bad(lv + "key out of range at voxel " + std::to_string(i));
            if (i > 0 && k <= prev) Bad(lv + (k == prev ? "duplicate key" : "keys not ascending") + " at voxel " + std::to_string(i));
            int x, y, z;
            unpack_voxel(k, x, y, z);
            if (x <= -lim || x >= lim || y <= -lim || y >= lim || z <= -lim || z >= lim)
                Bad(lv + "voxel coordinate outside +-2^20 at voxel " + std::to_string(i));
            prev = k;
            const uint32_t c = Get<uint32_t>(src + v.off_counts + 4 * i);
            if (c > (uint32_t) v.max_num_points)
                Bad(lv + "count " + std::to_string(c) + " > max_num_points at voxel " + std::to_string(i));
            sum += c;
        }
        if (sum != v.P) Bad(lv + "P = " + std::to_string(v.P) + " but the counts add up to " + std::to_string(sum));
        // a point's |w| - 1 indexes the frame origins (the normals' orientation): keep it inside frame_count
        for (uint64_t j = 0; j < v.P; ++j) {
            const float w = Get<float>(src + v.off_points + 16 * j + 12);
            const float a = std::fabs(w);
            if (!(a >= 1.f && a <= (float) L.frame_count && a == std::floor(a)))
                Bad(lv + "point " + std::to_string(j) + " has frame ordinal w = " + std::to_string(w));
        }
    }
    return L;
}

// ---- options ----
cticp_odometry_options CanonicalOptions(const cticp_odometry_options &o) {
    cticp_odometry_options c = o;
    c.map_options._pad0 = 0;
    for (auto &r : c.map_options.resolutions) r._pad0 = 0;
    c.neighborhood_strategy._pad0 = 0;
    c.adaptive_options._pad0 = 0;
    return c;
}

std::string FirstOptionDifference(const cticp_odometry_options &a0, const cticp_odometry_options &b0) {
    const cticp_odometry_options a = CanonicalOptions(a0), b = CanonicalOptions(b0);
    struct Field {
        const char *name;
        size_t offset, size;
    };
#define F(f) Field{#f, offsetof(cticp_odometry_options, f), sizeof(((cticp_odometry_options *) nullptr)->f)}
    static const Field fields[] = {
        F(ct_icp_options.num_iters_icp), F(ct_icp_options.parametrization), F(ct_icp_options.distance),
        F(ct_icp_options.solver), F(ct_icp_options.max_num_residuals), F(ct_icp_options.min_num_residuals),
        F(ct_icp_options.weighting_scheme), F(ct_icp_options.max_number_neighbors), F(ct_icp_options.min_number_neighbors),
        F(ct_icp_options.threshold_voxel_occupancy), F(ct_icp_options.num_closest_neighbors),
        F(ct_icp_options.point_to_plane_with_distortion), F(ct_icp_options.loss_function), F(ct_icp_options.ls_max_num_iters),
        F(ct_icp_options.ls_num_threads), F(ct_icp_options.debug_print), F(ct_icp_options.weight_alpha),
        F(ct_icp_options.weight_neighborhood), F(ct_icp_options.power_planarity), F(ct_icp_options.threshold_orientation_norm),
        F(ct_icp_options.threshold_translation_norm), F(ct_icp_options.ls_sigma), F(ct_icp_options.ls_tolerant_min_threshold),
        F(ct_icp_options.max_dist_to_plane_ct_icp), F(ct_icp_options.threshold_linearity), F(ct_icp_options.threshold_planarity),
        F(ct_icp_options.weight_point_to_point), F(ct_icp_options.outlier_distance), F(ct_icp_options.use_barycenter),
        F(ct_icp_options.use_lines),
        F(map_options.num_resolutions), F(map_options.select_valid_normals_direction), F(map_options.max_frames_to_keep),
        F(map_options.default_radius), F(map_options.resolutions),
        F(neighborhood_strategy.type), F(neighborhood_strategy.max_num_neighbors), F(neighborhood_strategy.min_num_neighbors),
        F(neighborhood_strategy.distance_max), F(neighborhood_strategy.radius_min), F(neighborhood_strategy.radius_max),
        F(neighborhood_strategy.exponent),
        F(default_motion_model.model), F(default_motion_model.log_if_invalid), F(default_motion_model.beta_location_consistency),
        F(default_motion_model.beta_constant_velocity), F(default_motion_model.beta_small_velocity),
        F(default_motion_model.beta_orientation_consistency), F(default_motion_model.threshold_orientation_deg),
        F(default_motion_model.threshold_translation_diff),
        F(motion_compensation), F(initialization), F(init_num_frames), F(max_num_keypoints), F(sampling), F(quit_on_error),
        F(robust_minimal_level), F(robust_registration), F(robust_fail_early), F(robust_num_attempts),
        F(robust_num_attempts_when_rotation), F(robust_max_voxel_neighborhood), F(always_insert), F(do_no_insert),
        F(debug_print), F(with_default_motion_model), F(init_voxel_size), F(init_sample_voxel_size), F(sample_voxel_size),
        F(voxel_size), F(max_distance), F(distance_error_threshold), F(orientation_error_threshold),
        F(robust_full_voxel_threshold), F(robust_empty_voxel_threshold), F(robust_neighborhood_min_dist),
        F(robust_neighborhood_min_orientation), F(robust_relative_trans_threshold), F(robust_threshold_ego_orientation),
        F(robust_threshold_relative_orientation), F(insertion_ego_rotation_threshold), F(insertion_threshold_frames_skipped),
        F(insertion_cum_distance_threshold), F(insertion_cum_orientation_threshold), F(shuffle_seed),
        F(adaptive_options.num_points_per_voxel), F(adaptive_options.max_num_points), F(adaptive_options.num_bands),
        F(adaptive_options.distance), F(adaptive_options.voxel_size),
    };
#undef F
    const uint8_t *pa = reinterpret_cast<const uint8_t *>(&a), *pb = reinterpret_cast<const uint8_t *>(&b);
    for (const Field &f : fields)
        if (memcmp(pa + f.offset, pb + f.offset, f.size) != 0) return f.name;
    return "";
}

// ---- odometry blob ----
size_t OdoBlobSize(size_t trajectory_size, size_t map_size) {
    return kOdoHeaderBytes + Align8(sizeof(cticp_odometry_options)) + sizeof(OdoHostRecord) +
           sizeof(cticp_frame) * trajectory_size + map_size;
}

void OdoWrite(uint8_t *dst, const cticp_odometry_options &options, const OdoHostRecord &host, const cticp_frame *trajectory,
              size_t map_size) {
    const size_t total = OdoBlobSize(host.trajectory_size, map_size);
    memset(dst, 0, kOdoHeaderBytes + Align8(sizeof(cticp_odometry_options)));
    memcpy(dst, kOdoMagic, 8);
    Put<uint32_t>(dst + 8, kStateVersion);
    Put<uint32_t>(dst + 12, (uint32_t) sizeof(cticp_odometry_options));
    Put<uint64_t>(dst + 16, (uint64_t) total);
    size_t o = kOdoHeaderBytes;
    const cticp_odometry_options c = CanonicalOptions(options);
    memcpy(dst + o, &c, sizeof(c));
    o += Align8(sizeof(c));
    memcpy(dst + o, &host, sizeof(host));
    o += sizeof(host);
    if (host.trajectory_size) memcpy(dst + o, trajectory, sizeof(cticp_frame) * host.trajectory_size);
}

OdoBlobView OdoParse(const uint8_t *src, size_t size, bool full) {
    CheckHeader(src, size, kOdoMagic, "odometry blob");
    if (Get<uint32_t>(src + 12) != sizeof(cticp_odometry_options))
        Bad("options record of " + std::to_string(Get<uint32_t>(src + 12)) + " bytes (this build: " +
            std::to_string(sizeof(cticp_odometry_options)) + ")");
    const size_t fixed = OdoBlobSize(0, 0);
    if (size < fixed) Bad("odometry blob truncated");
    OdoBlobView v;
    memcpy(&v.options, src + kOdoHeaderBytes, sizeof(v.options));
    memcpy(&v.host, src + kOdoHeaderBytes + Align8(sizeof(cticp_odometry_options)), sizeof(v.host));
    v.trajectory = reinterpret_cast<const cticp_frame *>(src + fixed);
    v.map = nullptr;
    v.map_size = 0;
    if (!full) return v;
    const uint64_t T = v.host.trajectory_size;
    if (T > (size - fixed) / sizeof(cticp_frame)) Bad("trajectory of " + std::to_string(T) + " frames exceeds the blob");
    if (v.host.registered_frames < 0 || (uint64_t) v.host.registered_frames != T)
        Bad("registered_frames " + std::to_string(v.host.registered_frames) + " != trajectory size " + std::to_string(T));
    if (v.host.last_num_keypoints < 0) Bad("last_num_keypoints");
    v.map = src + fixed + sizeof(cticp_frame) * T;
    v.map_size = size - fixed - sizeof(cticp_frame) * T;
    return v;
}

}  // namespace cticp
