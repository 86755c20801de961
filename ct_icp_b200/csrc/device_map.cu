// device_map.cu — insert / evict / rebuild / export kernels and the host-side DeviceMap class.
//
// Reference behaviour reproduced (include/ct_icp/map.h):
//   InsertPointCloud / InsertPointInVoxelMap  :153-254, 261-293  (sequential min-distance rule in input order)
//   RemoveElementsFarFromLocation             :305-322           (tests the voxel's FIRST stored point)
//   NumPoints / GetMapPoints                  :345-376
#include "device_map.h"

#include <cooperative_groups.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "gather.cuh"
#include "frame_policy.h"
#include "state_io.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>
#include <vector>

namespace cticp {

#define CT_CUDA_CHECK(expr)                                                                              \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            throw CudaError(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                            std::to_string(__LINE__));                                                   \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------
__global__ void k_clear_level(MapLevel L) {
    const uint32_t cap = L.cap_mask + 1;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
        L.slots[i].key = kEmptyKey;
        L.slots[i].count = 0;
        L.slots[i]._pad = 0;
        L.head[i] = kNil;
        if (L.normals) L.normals[4 * (size_t) i + 3] = 0.0;
    }
}

// Phase 1 of InsertPointCloud: find-or-create the voxel of every point and thread the point onto the voxel's
// candidate list. One thread per point; the list order is arbitrary (phase 2 re-orders by point index).
// A voxel that already holds B points accepts nothing (map.h:276-291) and its count only changes in phase 2, so its
// points are neither threaded nor is the voxel touched: phase 2 only visits voxels that can still change.
__device__ __forceinline__ void insert_claim_dev(const MapLevel &L, MapCounters *ctr, const double *world, int n,
                                                 int *__restrict__ next, uint32_t *__restrict__ touched) {
    const double inv_res = 1.0 / L.res;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double px = world[3 * i], py = world[3 * i + 1], pz = world[3 * i + 2];
        if (!(isfinite(px) && isfinite(py) && isfinite(pz))) {
            next[i] = kNil;
            continue;
        }
        const unsigned long long key =
            pack_voxel(voxel_coord_rcp(px, L.res, inv_res), voxel_coord_rcp(py, L.res, inv_res), voxel_coord_rcp(pz, L.res, inv_res));
        uint32_t h = hash_key(key) & L.cap_mask;
        int slot = -1;
        for (uint32_t probe = 0; probe <= L.cap_mask; ++probe) {
            unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(&L.slots[h].key);
            if (k == kEmptyKey) {
                k = atomicCAS(&L.slots[h].key, kEmptyKey, key);
                if (k == kEmptyKey) {
                    atomicAdd(&ctr->num_voxels, 1u);
                    slot = (int) h;
                    break;
                }
            }
            if (k == key) {
                slot = (int) h;
                break;
            }
            h = (h + 1) & L.cap_mask;
        }
        if (slot < 0) {
            atomicExch(&ctr->overflow, 1u);
            next[i] = kNil;
            continue;
        }
        if (L.slots[slot].count >= (uint32_t) L.B) {
            next[i] = kNil;
            continue;
        }
        const int old = atomicExch(&L.head[slot], i);
        next[i] = old;
        if (old == kNil) touched[atomicAdd(&ctr->num_touched, 1u)] = (uint32_t) slot;
    }
}
__global__ void k_insert_claim(MapLevel L, MapCounters *ctr, const double *__restrict__ world, const int *d_n,
                               int *__restrict__ next, uint32_t *__restrict__ touched) {
    insert_claim_dev(L, ctr, world, *d_n, next, touched);
}

// Phase 2: one warp per touched voxel applies the reference's sequential rule to that voxel's candidates in
// ascending point index: accept while count < B and every stored point is farther than min_dist (map.h:276-291);
// a brand-new voxel accepts its first candidate unconditionally (:268-273).
constexpr int kInsertWarps = 4;
constexpr int kMaxCand = 512;
constexpr int kMaxB = 64;

__device__ __forceinline__ double commit_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct CommitScratch {
    int cand[kInsertWarps][kMaxCand];
    int sorted[kInsertWarps][kMaxCand];
    float4 pts[kInsertWarps][kMaxB];
};
__device__ __forceinline__ void insert_commit_dev(const MapLevel &L, MapCounters *ctr, const double *world,
                                                  const int *next, const uint32_t *touched, const double *frame_origins,
                                                  int frame_ordinal, CommitScratch &sc) {
    int (&s_cand)[kInsertWarps][kMaxCand] = sc.cand;
    int (&s_sorted)[kInsertWarps][kMaxCand] = sc.sorted;
    float4 (&s_pts)[kInsertWarps][kMaxB] = sc.pts;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned n_touched = *reinterpret_cast<volatile unsigned *>(&ctr->num_touched);
    const int warps_total = gridDim.x * kInsertWarps;
    for (unsigned t = blockIdx.x * kInsertWarps + w; t < n_touched; t += warps_total) {
        const uint32_t slot = touched[t];
        const unsigned long long key = L.slots[slot].key;
        int vx, vy, vz;
        unpack_voxel(key, vx, vy, vz);
        const double ox = vx * L.res, oy = vy * L.res, oz = vz * L.res;
        const int count0 = (int) L.slots[slot].count;
        int count = count0;
        float4 *gpts = L.points + (size_t) slot * L.B;
        for (int j = lane; j < count; j += 32) s_pts[w][j] = gpts[j];

        // walk the candidate list (all lanes follow the same pointers → broadcast loads)
        int n = 0;
        for (int c = L.head[slot]; c != kNil; c = next[c]) {
            if (n < kMaxCand && lane == 0) s_cand[w][n] = c;
            ++n;
        }
        __syncwarp();
        int last = -1;          // slow path cursor (n > kMaxCand)
        int processed = 0;
        while (processed < n && count < L.B) {
            int m;              // candidates staged in s_sorted this round
            if (n <= kMaxCand) {
                // rank sort (indices are unique)
                for (int a = lane; a < n; a += 32) {
                    const int v = s_cand[w][a];
                    int rank = 0;
                    for (int b = 0; b < n; ++b) rank += (s_cand[w][b] < v);
                    s_sorted[w][rank] = v;
                }
                m = n;
            } else {
                // rare: more candidates than staging room → select the next smallest index by walking the list
                int best = 0x7fffffff;
                for (int c = L.head[slot]; c != kNil; c = next[c])
                    if (c > last && c < best) best = c;
                if (lane == 0) s_sorted[w][0] = best;
                last = best;
                m = 1;
            }
            __syncwarp();
            for (int a0 = 0; a0 < m && count < L.B; a0 += 32) {
                // the local coordinates of the next 32 candidates, loaded by the lanes side by side: the sequential rule
                // below then waits on no global load
                double cx = 0.0, cy = 0.0, cz = 0.0;
                if (a0 + lane < m) {
                    const int c = s_sorted[w][a0 + lane];
                    cx = world[3 * c] - ox; cy = world[3 * c + 1] - oy; cz = world[3 * c + 2] - oz;
                }
                const int chunk = min(32, m - a0);
                for (int a = 0; a < chunk && count < L.B; ++a) {
                    const double lx = __shfl_sync(0xffffffffu, cx, a), ly = __shfl_sync(0xffffffffu, cy, a),
                                 lz = __shfl_sync(0xffffffffu, cz, a);
                    bool too_close = false;
                    for (int j = lane; j < count; j += 32) {
                        const float4 q = s_pts[w][j];
                        const double dx = (double) q.x - lx, dy = (double) q.y - ly, dz = (double) q.z - lz;
                        const double d2 = dx * dx + dy * dy + dz * dz;
                        too_close |= !(d2 > L.min_dist2);
                    }
                    const bool reject = __any_sync(0xffffffffu, too_close);
                    if (!reject) {
                        if (lane == 0) {
                            const float4 v = make_float4((float) lx, (float) ly, (float) lz, (float) (frame_ordinal + 1));
                            s_pts[w][count] = v;
                            gpts[count] = v;
                        }
                        ++count;
                    }
                    __syncwarp();
                }
            }
            processed += m;
        }
        if (lane == 0) {
            L.slots[slot].count = (uint32_t) count;
            L.head[slot] = kNil;
            if (count > count0) atomicAdd(&ctr->num_points, (unsigned long long) (count - count0));
        }
        __syncwarp();
        // map.h:211-235: a voxel that received a point and holds >= 5 gets the normal of ALL its points (V.col(2) of
        // their covariance), copied to every point and oriented point by point against the begin position of the frame
        // that point came from. The sign lives in the sign of the point's w.
        if (L.normals && count > count0 && count >= 5) {
            double sx = 0, sy = 0, sz = 0, sxx = 0, sxy = 0, sxz = 0, syy = 0, syz = 0, szz = 0;
            for (int j = lane; j < count; j += 32) {
                const float4 q = s_pts[w][j];
                const double x = (double) q.x, y = (double) q.y, z = (double) q.z;   // relative to the voxel origin
                sx += x; sy += y; sz += z;
                sxx += x * x; sxy += x * y; sxz += x * z; syy += y * y; syz += y * z; szz += z * z;
            }
            const double inv = 1.0 / (double) count;
            const double mx = commit_warp_sum(sx) * inv, my = commit_warp_sum(sy) * inv, mz = commit_warp_sum(sz) * inv;
            const double cxx = commit_warp_sum(sxx) * inv - mx * mx, cxy = commit_warp_sum(sxy) * inv - mx * my,
                         cxz = commit_warp_sum(sxz) * inv - mx * mz, cyy = commit_warp_sum(syy) * inv - my * my,
                         cyz = commit_warp_sum(syz) * inv - my * mz, czz = commit_warp_sum(szz) * inv - mz * mz;
            const Eig3 e = sym_eig3(cxx, cxy, cxz, cyy, cyz, czz);
            if (lane == 0) {
                double *nrm = L.normals + 4 * (size_t) slot;
                nrm[0] = e.normal.x; nrm[1] = e.normal.y; nrm[2] = e.normal.z; nrm[3] = 1.0;
            }
            for (int j = lane; j < count; j += 32) {
                float4 q = s_pts[w][j];
                const int f = (int) fabsf(q.w) - 1;
                const double px = ox + (double) q.x - frame_origins[3 * f], py = oy + (double) q.y - frame_origins[3 * f + 1],
                             pz = oz + (double) q.z - frame_origins[3 * f + 2];
                const bool flip = px * e.normal.x + py * e.normal.y + pz * e.normal.z > 0.0;
                q.w = flip ? -fabsf(q.w) : fabsf(q.w);
                gpts[j] = q;
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kInsertWarps * 32)
k_insert_commit(MapLevel L, MapCounters *ctr, const double *__restrict__ world, const int *__restrict__ next,
                const uint32_t *__restrict__ touched, const double *__restrict__ frame_origins, int frame_ordinal) {
    __shared__ CommitScratch sc;
    insert_commit_dev(L, ctr, world, next, touched, frame_origins, frame_ordinal, sc);
}

// RemoveElementsFarFromLocation (map.h:305-322): a voxel goes when its FIRST stored point is farther than
// `distance` from `location` (or when it is empty). Tombstones keep probe chains intact; Rebuild() purges them.
__device__ __forceinline__ void remove_far_dev(const MapLevel &L, MapCounters *ctr, V3 loc, double distance) {
    const uint32_t cap = L.cap_mask + 1;
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += gridDim.x * blockDim.x) {
        const unsigned long long key = L.slots[s].key;
        if (key == kEmptyKey || key == kTombKey) continue;
        const uint32_t count = L.slots[s].count;
        bool remove = (count == 0);
        if (!remove) {
            int vx, vy, vz;
            unpack_voxel(key, vx, vy, vz);
            const float4 p = L.points[(size_t) s * L.B];
            const double dx = vx * L.res + (double) p.x - loc.x, dy = vy * L.res + (double) p.y - loc.y,
                         dz = vz * L.res + (double) p.z - loc.z;
            remove = sqrt(dx * dx + dy * dy + dz * dz) > distance;
        }
        if (remove) {
            L.slots[s].key = kTombKey;
            L.slots[s].count = 0;
            atomicAdd(&ctr->num_tombs, 1u);
            atomicSub(&ctr->num_voxels, 1u);
            atomicAdd(&ctr->num_points, (unsigned long long) (-(long long) count));
        }
    }
}

__global__ void k_remove_far(MapLevel L, MapCounters *ctr, V3 loc, double distance) { remove_far_dev(L, ctr, loc, distance); }

// ---- the whole map update of a frame (odometry.cpp:855-953: transform of the sub-sampled frame with the final pose pair,
// RemoveElementsFarFromLocation, InsertPointCloud on every resolution) in ONE cooperative launch: phases separated by
// grid barriers instead of 2 + 2 x levels kernels and their memsets (29 us of a 310 us step in round 1, most of it the
// fixed cost of five short dependent launches).
struct FusedUpdateArgs {
    MapLevel levels[CTICP_MAX_RESOLUTIONS];
    int num_levels;
    MapCounters *counters;
    const float4 *frame;        // sub-sampled frame (raw xyz, alpha)
    const float4 *frame_lo;     // its residual plane (nullptr: float32-representable, see load_raw)
    const int *d_n;
    double *world;              // out: its world points under the pose pair
    Q4 qb, qe;
    V3 tb, te;
    SlerpConsts sc;
    V3 location;                // eviction centre (the end position) and radius
    double max_distance;
    int do_remove, do_insert;
    int *next;
    uint32_t *touched;
    const double *frame_origins;
    int frame_ordinal;
    // speculative launch (frame_policy.h): pose pair, eviction centre and the evict / insert decision come from the verdict
    // k_frame_policy left on the device; the by-value fields above are then ignored
    const FrameVerdict *verdict;
    double *frame_origins_mut;
};
__global__ void __launch_bounds__(kInsertWarps * 32, 4)   // 4 co-resident CTAs per SM (UpdateFused's grid)
k_map_update_fused(FusedUpdateArgs a) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ CommitScratch sc;
    if (a.verdict) {
        const FrameVerdict &v = *a.verdict;
        const int action = v.action;
        if (action != kFrameEvict && action != kFrameInsert) return;   // uniform over the grid (before any barrier)
        a.qb = Q4{v.state.qb[0], v.state.qb[1], v.state.qb[2], v.state.qb[3]};
        a.qe = Q4{v.state.qe[0], v.state.qe[1], v.state.qe[2], v.state.qe[3]};
        a.tb = V3{v.state.tb[0], v.state.tb[1], v.state.tb[2]};
        a.te = V3{v.state.te[0], v.state.te[1], v.state.te[2]};
        a.sc = v.sc;
        a.location = a.te;   // trajectory_.back().end_pose.tr (odometry.cpp:942)
        a.do_insert = action == kFrameInsert;
        // frame_poses.front().tr of this insert (odometry.cpp:949); read by insert_commit_dev behind the grid barriers
        if (a.do_insert && a.frame_origins_mut && blockIdx.x == 0 && threadIdx.x == 0) {
            double *o = a.frame_origins_mut + 3 * (size_t) a.frame_ordinal;
            o[0] = a.tb.x; o[1] = a.tb.y; o[2] = a.tb.z;
        }
    }
    const int n = *a.d_n;
    // phase 1: world points of the frame; eviction on every level; reset the per-level touched counters
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const RawPoint p = load_raw(a.frame, a.frame_lo, i);
        const V3 w = ct_transform_c(a.qb, a.tb, a.qe, a.te, p.alpha, V3{p.x, p.y, p.z}, a.sc);
        a.world[3 * i] = w.x; a.world[3 * i + 1] = w.y; a.world[3 * i + 2] = w.z;
    }
    if (a.do_remove)
        for (int l = 0; l < a.num_levels; ++l) remove_far_dev(a.levels[l], a.counters + l, a.location, a.max_distance);
    if (blockIdx.x == 0 && threadIdx.x < a.num_levels) a.counters[threadIdx.x].num_touched = 0;
    if (!a.do_insert) return;   // uniform
    for (int l = 0; l < a.num_levels; ++l) {
        grid.sync();
        insert_claim_dev(a.levels[l], a.counters + l, a.world, n, a.next, a.touched);
        grid.sync();
        insert_commit_dev(a.levels[l], a.counters + l, a.world, a.next, a.touched, a.frame_origins, a.frame_ordinal, sc);
    }
}

// Find-or-create `key` in a table being filled from scratch (keys unique) and copy its run of `count` points and, when
// both sides keep them, its normal. Shared by the rebuild and by the load of a saved map.
__device__ __forceinline__ void place_voxel_dev(const MapLevel &dst, unsigned long long key, uint32_t count,
                                                const float4 *pts, const double *nrm) {
    uint32_t h = hash_key(key) & dst.cap_mask;
    for (uint32_t probe = 0; probe <= dst.cap_mask; ++probe) {
        if (atomicCAS(&dst.slots[h].key, kEmptyKey, key) == kEmptyKey) break;
        h = (h + 1) & dst.cap_mask;
    }
    dst.slots[h].count = count;
    for (uint32_t j = 0; j < count; ++j) dst.points[(size_t) h * dst.B + j] = pts[j];
    if (nrm && dst.normals)
        for (int c = 0; c < 4; ++c) dst.normals[4 * (size_t) h + c] = nrm[c];
}

// Re-hash the live voxels of `src` into the empty table `dst` (purges tombstones, optionally grows).
__global__ void k_rebuild(MapLevel src, MapLevel dst, MapCounters *ctr) {
    const uint32_t cap = src.cap_mask + 1;
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += gridDim.x * blockDim.x) {
        const unsigned long long key = src.slots[s].key;
        if (key == kEmptyKey || key == kTombKey) continue;
        place_voxel_dev(dst, key, src.slots[s].count, src.points + (size_t) s * src.B,
                        src.normals ? src.normals + 4 * (size_t) s : nullptr);
    }
    (void) ctr;
}

// ---- canonical order of a level (export, save): the live voxels compacted, sorted by packed key on the device, their
// point runs at the exclusive scan of the counts. Ascending packed key is lexicographic (x, y, z): the bias makes every
// 21-bit field non-negative. The compaction's order depends on atomic timing; the sort removes it.
// (`room` entries of output, the live-voxel counter: the host checks the final cursor against it)
__global__ void k_live_slots(MapLevel L, unsigned long long *keys, uint32_t *slots, unsigned room, unsigned int *cursor) {
    const uint32_t cap = L.cap_mask + 1;
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += gridDim.x * blockDim.x) {
        const unsigned long long key = L.slots[s].key;
        if (key == kEmptyKey || key == kTombKey) continue;
        const unsigned i = atomicAdd(cursor, 1u);
        if (i >= room) continue;
        keys[i] = key;
        slots[i] = s;
    }
}
__global__ void k_sorted_counts(MapLevel L, const uint32_t *__restrict__ slots, size_t V, uint32_t *counts,
                                unsigned long long *counts64) {
    for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < V; i += (size_t) gridDim.x * blockDim.x) {
        const uint32_t c = L.slots[slots[i]].count;
        counts[i] = c;
        counts64[i] = c;
    }
}
// one warp per voxel run: the dense point runs (and normals) of a save, in key order
__global__ void k_gather_runs(MapLevel L, const uint32_t *__restrict__ slots, const uint32_t *__restrict__ counts,
                              const unsigned long long *__restrict__ offsets, size_t V, float4 *out_pts, double *out_normals) {
    const int lane = threadIdx.x & 31;
    const size_t warps = (size_t) gridDim.x * (blockDim.x >> 5);
    for (size_t v = (blockIdx.x * (size_t) blockDim.x + threadIdx.x) >> 5; v < V; v += warps) {
        const size_t s = slots[v];
        const uint32_t c = counts[v];
        const unsigned long long o = offsets[v];
        for (uint32_t j = lane; j < c; j += 32) out_pts[o + j] = L.points[s * L.B + j];
        if (out_normals && lane < 4) out_normals[4 * v + lane] = L.normals[4 * s + lane];
    }
}
// one warp per voxel run: GetMapPoints as fp64 world xyz + voxel coordinates, in key order
__global__ void k_export_runs(MapLevel L, const unsigned long long *__restrict__ keys, const uint32_t *__restrict__ slots,
                              const uint32_t *__restrict__ counts, const unsigned long long *__restrict__ offsets, size_t V,
                              double *xyz, int *voxel) {
    const int lane = threadIdx.x & 31;
    const size_t warps = (size_t) gridDim.x * (blockDim.x >> 5);
    for (size_t v = (blockIdx.x * (size_t) blockDim.x + threadIdx.x) >> 5; v < V; v += warps) {
        int vx, vy, vz;
        unpack_voxel(keys[v], vx, vy, vz);
        const size_t s = slots[v];
        const uint32_t c = counts[v];
        const unsigned long long o0 = offsets[v];
        for (uint32_t j = lane; j < c; j += 32) {
            const unsigned long long o = o0 + j;
            const float4 p = L.points[s * L.B + j];
            xyz[3 * o] = vx * L.res + (double) p.x;
            xyz[3 * o + 1] = vy * L.res + (double) p.y;
            xyz[3 * o + 2] = vz * L.res + (double) p.z;
            voxel[3 * o] = vx; voxel[3 * o + 1] = vy; voxel[3 * o + 2] = vz;
        }
    }
}
__global__ void k_widen_counts(const uint32_t *__restrict__ counts, size_t V, unsigned long long *counts64) {
    for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < V; i += (size_t) gridDim.x * blockDim.x) counts64[i] = counts[i];
}
// load of a saved level into an empty table: one thread per voxel, like the rebuild
__global__ void k_place_runs(MapLevel dst, const unsigned long long *__restrict__ keys, const uint32_t *__restrict__ counts,
                             const unsigned long long *__restrict__ offsets, size_t V, const float4 *__restrict__ pts,
                             const double *__restrict__ normals) {
    for (size_t v = blockIdx.x * (size_t) blockDim.x + threadIdx.x; v < V; v += (size_t) gridDim.x * blockDim.x)
        place_voxel_dev(dst, keys[v], counts[v], pts + offsets[v], normals ? normals + 4 * v : nullptr);
}

// ---------------------------------------------------------------------------------------------------------------
static uint32_t NextPow2(uint64_t v) {
    uint64_t p = 1;
    while (p < v) p <<= 1;
    return (uint32_t) p;
}

DeviceMap::DeviceMap(const cticp_map_options &options, cudaStream_t stream, bool with_normals)
    : options_(options), stream_(stream), with_normals_(with_normals) {
    if (options.num_resolutions < 1 || options.num_resolutions > CTICP_MAX_RESOLUTIONS)
        throw std::invalid_argument("map_options.num_resolutions out of range");
    levels_.resize(options.num_resolutions);
    for (int i = 0; i < options.num_resolutions; ++i) {
        const auto &rp = options.resolutions[i];
        if (!(rp.resolution > 0) || rp.max_num_points < 1 || rp.max_num_points > kMaxB)
            throw std::invalid_argument("map resolution / max_num_points out of the supported range (1..64)");
        AllocLevel(levels_[i], (uint32_t) InitialCapacity(rp), rp);
    }
    CT_CUDA_CHECK(cudaMalloc(&d_counters_, sizeof(MapCounters) * levels_.size()));
    CT_CUDA_CHECK(cudaMemsetAsync(d_counters_, 0, sizeof(MapCounters) * levels_.size(), stream_));
    CT_CUDA_CHECK(cudaMalloc(&d_scalar_, 64));
    CT_CUDA_CHECK(cudaMallocHost(&h_counters_, sizeof(MapCounters) * CTICP_MAX_RESOLUTIONS));
    memset(h_counters_, 0, sizeof(MapCounters) * CTICP_MAX_RESOLUTIONS);
}

// default capacity: enough for a 100 m local map at load <= 0.5; tables double on demand (MaintainTables)
uint64_t DeviceMap::InitialCapacity(const cticp_resolution_param &rp) const {
    const uint64_t cap = options_.capacity_voxels ? options_.capacity_voxels : (rp.resolution < 0.5 ? (1ull << 20) : (1ull << 18));
    return NextPow2(std::max<uint64_t>(cap, 1024));
}

DeviceMap::~DeviceMap() {
    for (auto &L : levels_) FreeLevel(L);
    cudaFree(d_counters_);
    cudaFree(d_scalar_);
    cudaFree(d_next_);
    cudaFree(d_touched_);
    cudaFree(d_world_tmp_);
    cudaFree(d_frame_origins_);
    cudaFreeHost(h_counters_);
}

void DeviceMap::AllocLevel(MapLevel &L, uint32_t cap, const cticp_resolution_param &rp) {
    L.cap_mask = cap - 1;
    L.B = rp.max_num_points;
    L.res = rp.resolution;
    L.min_dist2 = rp.min_distance_between_points * rp.min_distance_between_points;
    CT_CUDA_CHECK(cudaMalloc(&L.slots, sizeof(MapSlot) * (size_t) cap));
    CT_CUDA_CHECK(cudaMalloc(&L.points, sizeof(float4) * (size_t) cap * L.B));
    CT_CUDA_CHECK(cudaMalloc(&L.head, sizeof(int) * (size_t) cap));
    L.normals = nullptr;
    if (with_normals_) CT_CUDA_CHECK(cudaMalloc(&L.normals, sizeof(double) * 4 * (size_t) cap));
    k_clear_level<<<592, 256, 0, stream_>>>(L);
    CT_CUDA_CHECK(cudaGetLastError());
}
void DeviceMap::FreeLevel(MapLevel &L) {
    cudaFree(L.slots);
    cudaFree(L.points);
    cudaFree(L.head);
    cudaFree(L.normals);
    L.normals = nullptr;
    L.slots = nullptr;
    L.points = nullptr;
    L.head = nullptr;
}

void DeviceMap::EnsureScratch(size_t n_upper) {
    if (n_upper <= scratch_n_) return;
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    cudaFree(d_next_);
    cudaFree(d_touched_);
    size_t n = std::max<size_t>(n_upper, 1024);
    CT_CUDA_CHECK(cudaMalloc(&d_next_, sizeof(int) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_touched_, sizeof(uint32_t) * n));
    scratch_n_ = n;
}

void DeviceMap::InsertDevice(const double *d_world_xyz, const int *d_n, size_t n_upper, V3 origin) {
    if (n_upper == 0) return;
    EnsureScratch(n_upper);
    // frame_id_to_frame[fidx].poses.front() (map.h:158-160): one begin position per inserted frame, never erased
    if (frame_count_ >= (1u << 24) - 2) throw CapacityError("more than 2^24 frames inserted into one map");
    if (with_normals_) {
        if (frame_count_ >= frame_capacity_) {
            const size_t cap = std::max<size_t>(4096, frame_capacity_ * 2);
            double *fresh = nullptr;
            CT_CUDA_CHECK(cudaMalloc(&fresh, sizeof(double) * 3 * cap));
            if (frame_count_)
                CT_CUDA_CHECK(cudaMemcpyAsync(fresh, d_frame_origins_, sizeof(double) * 3 * frame_count_,
                                              cudaMemcpyDeviceToDevice, stream_));
            CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
            cudaFree(d_frame_origins_);
            d_frame_origins_ = fresh;
            frame_capacity_ = cap;
        }
        // 24 bytes by value through a kernel-free path: cudaMemcpyAsync from pageable memory copies the source before
        // returning, so the stack variable may go out of scope
        const double o[3] = {origin.x, origin.y, origin.z};
        CT_CUDA_CHECK(cudaMemcpyAsync(d_frame_origins_ + 3 * frame_count_, o, sizeof(o), cudaMemcpyHostToDevice, stream_));
    }
    const int frame_ordinal = (int) frame_count_++;
    const int threads = 256;
    const int blocks = (int) std::min<size_t>((n_upper + threads - 1) / threads, 148 * 8);
    for (size_t i = 0; i < levels_.size(); ++i) {
        MapCounters *ctr = d_counters_ + i;
        CT_CUDA_CHECK(cudaMemsetAsync(&ctr->num_touched, 0, sizeof(unsigned), stream_));
        k_insert_claim<<<blocks, threads, 0, stream_>>>(levels_[i], ctr, d_world_xyz, d_n, d_next_, d_touched_);
        const int cblocks = (int) std::min<size_t>((n_upper + kInsertWarps - 1) / kInsertWarps, 148 * 8);
        k_insert_commit<<<cblocks, kInsertWarps * 32, 0, stream_>>>(levels_[i], ctr, d_world_xyz, d_next_, d_touched_,
                                                                     d_frame_origins_, frame_ordinal);
        launches_ += 2;
    }
    CT_CUDA_CHECK(cudaGetLastError());
    dirty_ = true;
}

void DeviceMap::EnsureFrameOrigin() {
    if (frame_count_ >= (1u << 24) - 2) throw CapacityError("more than 2^24 frames inserted into one map");
    if (with_normals_ && frame_count_ >= frame_capacity_) {
        const size_t cap = std::max<size_t>(4096, frame_capacity_ * 2);
        double *fresh = nullptr;
        CT_CUDA_CHECK(cudaMalloc(&fresh, sizeof(double) * 3 * cap));
        if (frame_count_)
            CT_CUDA_CHECK(cudaMemcpyAsync(fresh, d_frame_origins_, sizeof(double) * 3 * frame_count_,
                                          cudaMemcpyDeviceToDevice, stream_));
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        cudaFree(d_frame_origins_);
        d_frame_origins_ = fresh;
        frame_capacity_ = cap;
    }
}

void DeviceMap::UpdateFused(const float4 *d_frame, const float4 *d_frame_lo, const int *d_n, size_t n_upper, double *d_world, const Q4 &qb,
                            const V3 &tb, const Q4 &qe, const V3 &te, bool do_remove, V3 location, double max_distance,
                            bool do_insert, V3 origin, const FrameVerdict *d_verdict) {
    if (n_upper == 0) return;
    EnsureScratch(n_upper);
    int frame_ordinal = 0;
    if (d_verdict) {
        // speculative: whether this launch inserts is decided on the device; the slot of the frame's origin is reserved
        // now and kept by CommitSpeculativeInsert(true)
        EnsureFrameOrigin();
        frame_ordinal = (int) frame_count_;
    } else if (do_insert) {
        EnsureFrameOrigin();
        if (with_normals_) {
            const double o[3] = {origin.x, origin.y, origin.z};
            CT_CUDA_CHECK(cudaMemcpyAsync(d_frame_origins_ + 3 * frame_count_, o, sizeof(o), cudaMemcpyHostToDevice, stream_));
        }
        frame_ordinal = (int) frame_count_++;
    }
    if (fused_grid_ == 0) {
        int per_sm = 0, dev = 0, sms = 148;
        CT_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_map_update_fused, kInsertWarps * 32, 0));
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        int want = 4;   // CTAs per SM: more hide the latency of the probes, fewer make the grid barriers cheaper (A/B knob)
        if (const char *e = getenv("CTICP_UPDATE_CTAS_PER_SM")) want = std::max(1, atoi(e));
        fused_grid_ = std::max(1, std::min(per_sm, want) * sms);
    }
    FusedUpdateArgs a{};
    a.num_levels = (int) levels_.size();
    for (int l = 0; l < a.num_levels; ++l) a.levels[l] = levels_[l];
    a.counters = d_counters_;
    a.frame = d_frame;
    a.frame_lo = d_frame_lo;
    a.d_n = d_n;
    a.world = d_world;
    a.qb = qb; a.qe = qe; a.tb = tb; a.te = te;
    a.sc = slerp_consts(qb, qe);
    a.location = location;
    a.max_distance = max_distance;
    a.do_remove = do_remove ? 1 : 0;
    a.do_insert = do_insert ? 1 : 0;
    a.next = d_next_;
    a.touched = d_touched_;
    a.frame_origins = d_frame_origins_;
    a.frame_ordinal = frame_ordinal;
    a.verdict = d_verdict;
    a.frame_origins_mut = with_normals_ ? d_frame_origins_ : nullptr;
    void *args[] = {&a};
    CT_CUDA_CHECK(cudaLaunchCooperativeKernel((void *) k_map_update_fused, dim3(fused_grid_), dim3(kInsertWarps * 32), args, 0, stream_));
    launches_ += 1;
    dirty_ = true;
}

void DeviceMap::InsertHost(const double *xyz, size_t stride_bytes, size_t n, V3 origin) {
    if (n == 0) return;
    std::vector<double> packed(3 * n);
    for (size_t i = 0; i < n; ++i) {
        const double *p = reinterpret_cast<const double *>(reinterpret_cast<const char *>(xyz) + stride_bytes * i);
        packed[3 * i] = p[0]; packed[3 * i + 1] = p[1]; packed[3 * i + 2] = p[2];
    }
    SyncCounters();
    EnsureRoomFor(n);
    if (n > world_tmp_n_) {
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        cudaFree(d_world_tmp_);
        CT_CUDA_CHECK(cudaMalloc(&d_world_tmp_, sizeof(double) * 3 * n));
        world_tmp_n_ = n;
    }
    CT_CUDA_CHECK(cudaMemcpyAsync(d_world_tmp_, packed.data(), sizeof(double) * 3 * n, cudaMemcpyHostToDevice, stream_));
    int ni = (int) n;
    CT_CUDA_CHECK(cudaMemcpyAsync(d_scalar_, &ni, sizeof(int), cudaMemcpyHostToDevice, stream_));
    InsertDevice(d_world_tmp_, reinterpret_cast<int *>(d_scalar_), n, origin);
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));   // `packed` / `ni` go out of scope
    CheckOverflow();
}

void DeviceMap::RemoveFar(V3 location, double distance) {
    for (size_t i = 0; i < levels_.size(); ++i) {
        k_remove_far<<<592, 256, 0, stream_>>>(levels_[i], d_counters_ + i, location, distance);
        launches_ += 1;
    }
    CT_CUDA_CHECK(cudaGetLastError());
    dirty_ = true;
}

void DeviceMap::Clear() {
    for (auto &L : levels_) k_clear_level<<<592, 256, 0, stream_>>>(L);
    CT_CUDA_CHECK(cudaMemsetAsync(d_counters_, 0, sizeof(MapCounters) * levels_.size(), stream_));
    CT_CUDA_CHECK(cudaGetLastError());
    frame_count_ = 0;
    dirty_ = true;
}

const MapCounters *DeviceMap::SyncCounters() {
    if (dirty_) {
        CT_CUDA_CHECK(cudaMemcpyAsync(h_counters_, d_counters_, sizeof(MapCounters) * levels_.size(),
                                      cudaMemcpyDeviceToHost, stream_));
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        dirty_ = false;
        readback_pending_ = false;
    } else if (readback_pending_) {
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        readback_pending_ = false;
    }
    return h_counters_;
}

void DeviceMap::QueueCounterReadback() {
    CT_CUDA_CHECK(cudaMemcpyAsync(h_counters_, d_counters_, sizeof(MapCounters) * levels_.size(),
                                  cudaMemcpyDeviceToHost, stream_));
    dirty_ = false;   // valid after the next stream synchronisation
    readback_pending_ = true;
}

void DeviceMap::CheckOverflow() {
    const MapCounters *c = SyncCounters();
    for (size_t i = 0; i < levels_.size(); ++i)
        if (c[i].overflow) throw CapacityError("voxel table of map level " + std::to_string(i) + " is full");
}

// Purge tombstones / grow. Called by the odometry between frames with counters it already read back.
void DeviceMap::RebuildLevel(size_t i, uint64_t new_cap) {
    MapLevel fresh{};
    cticp_resolution_param rp = options_.resolutions[i];
    AllocLevel(fresh, (uint32_t) new_cap, rp);
    k_rebuild<<<592, 256, 0, stream_>>>(levels_[i], fresh, d_counters_ + i);
    CT_CUDA_CHECK(cudaMemsetAsync(&(d_counters_ + i)->num_tombs, 0, sizeof(unsigned), stream_));
    CT_CUDA_CHECK(cudaMemsetAsync(&(d_counters_ + i)->overflow, 0, sizeof(unsigned), stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    FreeLevel(levels_[i]);
    levels_[i] = fresh;
    h_counters_[i].num_tombs = 0;
    h_counters_[i].overflow = 0;
    ++rebuilds_;
}

void DeviceMap::MaintainTables() {
    const MapCounters *c = h_counters_;
    for (size_t i = 0; i < levels_.size(); ++i) {
        const uint64_t cap = (uint64_t) levels_[i].cap_mask + 1;
        const uint64_t used = (uint64_t) c[i].num_voxels + c[i].num_tombs;
        if (c[i].overflow) {
            // A probe sequence wrapped during the last insert: the points of that voxel were dropped (EnsureRoomFor makes
            // this unreachable for callers that announce their insert size). Recover — double the table, clear the flag —
            // and report the loss ONCE; the handle stays usable.
            RebuildLevel(i, cap * 2);
            throw CapacityError("voxel table of map level " + std::to_string(i) + " was full: points of the last insert were "
                                "dropped; the table has been doubled");
        }
        const bool grow = (uint64_t) c[i].num_voxels * 2 > cap;          // live load factor > 0.5
        const bool purge = used * 10 > cap * 7 || c[i].num_tombs * 4ull > cap;   // probe chains getting long
        if (!grow && !purge) continue;
        RebuildLevel(i, grow ? cap * 2 : cap);
    }
}

// Before an insert of up to n_new points (every one of them may open a new voxel): make sure no probe sequence can wrap.
// Uses the host copy of the counters (the previous frame's read-back), so it costs nothing unless a table must grow.
void DeviceMap::EnsureRoomFor(size_t n_new) {
    const MapCounters *c = h_counters_;
    for (size_t i = 0; i < levels_.size(); ++i) {
        uint64_t cap = (uint64_t) levels_[i].cap_mask + 1;
        const uint64_t live = (uint64_t) c[i].num_voxels + n_new, used = live + c[i].num_tombs;
        if (used * 10 <= cap * 8) continue;
        while (live * 2 > cap) cap *= 2;   // load <= 0.5 after the insert; tombstones vanish in the rebuild
        RebuildLevel(i, cap);
    }
}

void DeviceMap::SearchParams(double radius, int *level, int *voxel_neighborhood) const {
    // SearchParamsFromRadiusSearch, map.h:416-432
    int it = 0;
    while (it < options_.num_resolutions && options_.resolutions[it].resolution <= radius) ++it;
    int idx = std::max(0, it - 1);
    *level = idx;
    *voxel_neighborhood = (int) std::ceil(radius / options_.resolutions[idx].resolution);
}

// ---- canonical order, save, load ---------------------------------------------------------------------------------
template <typename T>
struct DeviceBuffer {   // scratch of one call, stream-ordered: no device-wide synchronisation on allocation or release
    T *p = nullptr;
    cudaStream_t stream;
    DeviceBuffer(size_t n, cudaStream_t s) : stream(s) {
        CT_CUDA_CHECK(cudaMallocAsync((void **) &p, sizeof(T) * std::max<size_t>(n, 1), stream));
    }
    ~DeviceBuffer() { cudaFreeAsync(p, stream); }
    DeviceBuffer(const DeviceBuffer &) = delete;
    DeviceBuffer &operator=(const DeviceBuffer &) = delete;
};

static int GridFor(size_t n, int threads) { return (int) std::max<size_t>(1, std::min<size_t>((n + threads - 1) / threads, 148 * 8)); }

// offsets[i] = counts[0] + ... + counts[i - 1] (counts64: the counts widened to 64 bit); returns the total (synchronises)
static uint64_t ExclusiveScan(const unsigned long long *counts64, const uint32_t *counts, unsigned long long *offsets, size_t V,
                              cudaStream_t stream) {
    if (V == 0) return 0;
    size_t tmp_bytes = 0;
    CT_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts64, offsets, (int) V, stream));
    DeviceBuffer<uint8_t> tmp(tmp_bytes, stream);
    CT_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, counts64, offsets, (int) V, stream));
    unsigned long long last_off = 0;
    uint32_t last_count = 0;
    CT_CUDA_CHECK(cudaMemcpyAsync(&last_off, offsets + V - 1, sizeof(last_off), cudaMemcpyDeviceToHost, stream));
    CT_CUDA_CHECK(cudaMemcpyAsync(&last_count, counts + V - 1, sizeof(last_count), cudaMemcpyDeviceToHost, stream));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream));
    return last_off + last_count;
}

struct DeviceMap::SortedLevel {   // the live voxels of one level in ascending key order
    SortedLevel(size_t n, cudaStream_t s) : keys(n, s), slots(n, s), counts(n, s), counts64(n, s), offsets(n, s) {}
    DeviceBuffer<unsigned long long> keys;
    DeviceBuffer<uint32_t> slots, counts;
    DeviceBuffer<unsigned long long> counts64, offsets;
    size_t V = 0;
    uint64_t P = 0;
};

std::unique_ptr<DeviceMap::SortedLevel> DeviceMap::SortLevel(int level, size_t num_voxels) {
    const MapLevel &L = levels_[level];
    const size_t cap = (size_t) L.cap_mask + 1;
    auto S = std::make_unique<SortedLevel>(num_voxels, stream_);
    DeviceBuffer<unsigned long long> keys_in(num_voxels, stream_);
    DeviceBuffer<uint32_t> slots_in(num_voxels, stream_);
    DeviceBuffer<unsigned int> cursor(1, stream_);
    CT_CUDA_CHECK(cudaMemsetAsync(cursor.p, 0, sizeof(unsigned int), stream_));
    k_live_slots<<<GridFor(cap, 256), 256, 0, stream_>>>(L, keys_in.p, slots_in.p, (unsigned) num_voxels, cursor.p);
    CT_CUDA_CHECK(cudaGetLastError());
    unsigned int V = 0;
    CT_CUDA_CHECK(cudaMemcpyAsync(&V, cursor.p, sizeof(V), cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (V != num_voxels)
        throw std::runtime_error("map level " + std::to_string(level) + ": " + std::to_string(V) + " live voxels, the counter says " +
                                 std::to_string(num_voxels));
    S->V = V;
    if (V == 0) return S;
    size_t tmp_bytes = 0;
    // bit 63 of a packed key is always 0
    CT_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys_in.p, S->keys.p, slots_in.p, S->slots.p, (int) V, 0, 63,
                                                  stream_));
    DeviceBuffer<uint8_t> tmp(tmp_bytes, stream_);
    CT_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, keys_in.p, S->keys.p, slots_in.p, S->slots.p, (int) V, 0, 63,
                                                  stream_));
    k_sorted_counts<<<GridFor(V, 256), 256, 0, stream_>>>(L, S->slots.p, V, S->counts.p, S->counts64.p);
    CT_CUDA_CHECK(cudaGetLastError());
    S->P = ExclusiveScan(S->counts64.p, S->counts.p, S->offsets.p, V, stream_);
    return S;
}

size_t DeviceMap::Export(int level, std::vector<double> &xyz, std::vector<int> &voxels) {
    const MapCounters *c = SyncCounters();
    const size_t n = (size_t) c[level].num_points;
    xyz.assign(3 * n, 0.0);
    voxels.assign(3 * n, 0);
    if (n == 0) return 0;
    auto S = SortLevel(level, c[level].num_voxels);
    if (S->P != n) throw std::runtime_error("map level " + std::to_string(level) + ": the voxel runs hold " + std::to_string(S->P) +
                                            " points, the counter " + std::to_string(n));
    DeviceBuffer<double> d_xyz(3 * n, stream_);
    DeviceBuffer<int> d_vox(3 * n, stream_);
    k_export_runs<<<GridFor(32 * S->V, 256), 256, 0, stream_>>>(levels_[level], S->keys.p, S->slots.p, S->counts.p, S->offsets.p,
                                                                 S->V, d_xyz.p, d_vox.p);
    CT_CUDA_CHECK(cudaGetLastError());
    CT_CUDA_CHECK(cudaMemcpyAsync(xyz.data(), d_xyz.p, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaMemcpyAsync(voxels.data(), d_vox.p, sizeof(int) * 3 * n, cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    return n;
}

size_t DeviceMap::Save(uint8_t *dst, size_t cap) {
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    // the counters are read privately: the host copy MaintainTables works from stays what the last frame left
    std::vector<MapCounters> c(levels_.size());
    CT_CUDA_CHECK(cudaMemcpyAsync(c.data(), d_counters_, sizeof(MapCounters) * c.size(), cudaMemcpyDeviceToHost, stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    MapBlobLayout B;
    B.num_levels = (int) levels_.size();
    B.has_normals = with_normals_;
    B.frame_count = frame_count_;
    for (int l = 0; l < B.num_levels; ++l) {
        const auto &rp = options_.resolutions[l];
        B.levels[l].resolution = rp.resolution;
        B.levels[l].min_distance = rp.min_distance_between_points;
        B.levels[l].max_num_points = rp.max_num_points;
        B.levels[l].V = c[l].num_voxels;
        B.levels[l].P = c[l].num_points;
    }
    MapLayoutFill(B);
    if (!dst || cap < B.total) return B.total;
    if (with_normals_ && frame_count_)
        CT_CUDA_CHECK(cudaMemcpyAsync(dst + B.off_origins, d_frame_origins_, sizeof(double) * 3 * frame_count_,
                                      cudaMemcpyDeviceToHost, stream_));
    for (int l = 0; l < B.num_levels; ++l) {
        const MapBlobLevel &v = B.levels[l];
        auto S = SortLevel(l, v.V);
        if (S->P != v.P)
            throw std::runtime_error("map level " + std::to_string(l) + ": the voxel runs hold " + std::to_string(S->P) +
                                     " points, the counter says " + std::to_string(v.P));
        if (v.V == 0) continue;
        DeviceBuffer<float4> pts(v.P, stream_);
        DeviceBuffer<double> nrm(with_normals_ ? 4 * v.V : 0, stream_);
        k_gather_runs<<<GridFor(32 * v.V, 256), 256, 0, stream_>>>(levels_[l], S->slots.p, S->counts.p, S->offsets.p, v.V, pts.p,
                                                                    with_normals_ ? nrm.p : nullptr);
        CT_CUDA_CHECK(cudaGetLastError());
        CT_CUDA_CHECK(cudaMemcpyAsync(dst + v.off_keys, S->keys.p, 8 * v.V, cudaMemcpyDeviceToHost, stream_));
        CT_CUDA_CHECK(cudaMemcpyAsync(dst + v.off_counts, S->counts.p, 4 * v.V, cudaMemcpyDeviceToHost, stream_));
        if (v.P) CT_CUDA_CHECK(cudaMemcpyAsync(dst + v.off_points, pts.p, 16 * v.P, cudaMemcpyDeviceToHost, stream_));
        if (with_normals_) CT_CUDA_CHECK(cudaMemcpyAsync(dst + v.off_normals, nrm.p, 32 * v.V, cudaMemcpyDeviceToHost, stream_));
    }
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    MapWriteHeaders(dst, B);
    SealBlob(dst, B.total);
    return B.total;
}

void DeviceMap::Load(const uint8_t *src, size_t size) {
    const MapBlobLayout B = MapParse(src, size);
    if (B.num_levels != (int) levels_.size())
        throw std::invalid_argument("map load: the blob has " + std::to_string(B.num_levels) + " resolutions, this map " +
                                    std::to_string(levels_.size()));
    if (B.has_normals != with_normals_)
        throw std::invalid_argument(std::string("map load: the blob ") + (B.has_normals ? "keeps" : "does not keep") +
                                    " per-voxel normals, this map " + (with_normals_ ? "does" : "does not"));
    for (int l = 0; l < B.num_levels; ++l) {
        const auto &rp = options_.resolutions[l];
        const MapBlobLevel &v = B.levels[l];
        const std::string lv = "map load: resolutions[" + std::to_string(l) + "].";
        if (v.resolution != rp.resolution) throw std::invalid_argument(lv + "resolution differs");
        if (v.max_num_points != rp.max_num_points) throw std::invalid_argument(lv + "max_num_points differs");
        if (v.min_distance != rp.min_distance_between_points) throw std::invalid_argument(lv + "min_distance_between_points differs");
    }
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    // fresh tables at load factor <= 0.5 (MaintainTables' rule); the old ones are released only once all are placed
    std::vector<MapLevel> fresh(levels_.size(), MapLevel{});
    try {
        for (int l = 0; l < B.num_levels; ++l) {
            const MapBlobLevel &v = B.levels[l];
            uint64_t cap = InitialCapacity(options_.resolutions[l]);
            while (v.V * 2 > cap) cap *= 2;
            if (cap > (1ull << 31)) throw CapacityError("map load: more voxels than a table can hold");
            AllocLevel(fresh[l], (uint32_t) cap, options_.resolutions[l]);
            if (v.V == 0) continue;
            DeviceBuffer<unsigned long long> keys(v.V, stream_), counts64(v.V, stream_), offsets(v.V, stream_);
            DeviceBuffer<uint32_t> counts(v.V, stream_);
            DeviceBuffer<float4> pts(v.P, stream_);
            DeviceBuffer<double> nrm(with_normals_ ? 4 * v.V : 0, stream_);
            CT_CUDA_CHECK(cudaMemcpyAsync(keys.p, src + v.off_keys, 8 * v.V, cudaMemcpyHostToDevice, stream_));
            CT_CUDA_CHECK(cudaMemcpyAsync(counts.p, src + v.off_counts, 4 * v.V, cudaMemcpyHostToDevice, stream_));
            if (v.P) CT_CUDA_CHECK(cudaMemcpyAsync(pts.p, src + v.off_points, 16 * v.P, cudaMemcpyHostToDevice, stream_));
            if (with_normals_) CT_CUDA_CHECK(cudaMemcpyAsync(nrm.p, src + v.off_normals, 32 * v.V, cudaMemcpyHostToDevice, stream_));
            k_widen_counts<<<GridFor(v.V, 256), 256, 0, stream_>>>(counts.p, v.V, counts64.p);
            CT_CUDA_CHECK(cudaGetLastError());
            ExclusiveScan(counts64.p, counts.p, offsets.p, v.V, stream_);
            k_place_runs<<<GridFor(v.V, 256), 256, 0, stream_>>>(fresh[l], keys.p, counts.p, offsets.p, v.V, pts.p,
                                                                 with_normals_ ? nrm.p : nullptr);
            CT_CUDA_CHECK(cudaGetLastError());
        }
        if (with_normals_ && B.frame_count > frame_capacity_) {
            size_t fcap = std::max<size_t>(4096, frame_capacity_);
            while (fcap < B.frame_count) fcap *= 2;
            double *origins = nullptr;
            CT_CUDA_CHECK(cudaMalloc(&origins, sizeof(double) * 3 * fcap));
            cudaFree(d_frame_origins_);
            d_frame_origins_ = origins;
            frame_capacity_ = fcap;
        }
    } catch (...) {
        for (auto &L : fresh) FreeLevel(L);
        throw;
    }
    for (int l = 0; l < B.num_levels; ++l) {
        FreeLevel(levels_[l]);
        levels_[l] = fresh[l];
        MapCounters &c = h_counters_[l];
        c = MapCounters{};
        c.num_points = B.levels[l].P;
        c.num_voxels = (unsigned int) B.levels[l].V;
    }
    if (with_normals_ && B.frame_count)
        CT_CUDA_CHECK(cudaMemcpyAsync(d_frame_origins_, src + B.off_origins, sizeof(double) * 3 * B.frame_count,
                                      cudaMemcpyHostToDevice, stream_));
    CT_CUDA_CHECK(cudaMemcpyAsync(d_counters_, h_counters_, sizeof(MapCounters) * levels_.size(), cudaMemcpyHostToDevice, stream_));
    CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
    frame_count_ = B.frame_count;
    dirty_ = false;
    readback_pending_ = false;
}

}  // namespace cticp
