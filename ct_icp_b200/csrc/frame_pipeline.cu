// frame_pipeline.cu — per-scan device pipeline around the ICP: ingest, voxel sub-sampling, keypoint grid sampling,
// continuous-time transform of the frame.
//
// Reference: Odometry::InitializeFrame (src/ct_icp/odometry.cpp:333-382), sub_sample_frame / grid_sampling
// (src/ct_icp/ct_icp.cpp:65-101), the post-registration transforms (odometry.cpp:463-486).
//
// Order contract (DESIGN.md): std::shuffle + "first point seen per voxel" becomes
//   winner(voxel) = argmin over the voxel's points of perm(i)        [64-bit atomicMin on (perm(i) << 32 | i)]
//   output order  = ascending perm(i) of the winners                   [flag array in permuted index space + scan]
// and the second shuffle is one scatter through a second permutation — no sort anywhere.
#include "frame_pipeline.h"

#include <cooperative_groups.h>
#include <cstdlib>

#include <algorithm>
#include <cstring>

namespace cticp {

#define CT_CUDA_CHECK(expr)                                                                              \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            throw CudaError(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                            std::to_string(__LINE__));                                                   \
    } while (0)

constexpr unsigned long long kGridEmpty = ~0ull;
constexpr size_t kMaxTiles = 4096;   // up to 4M points per scan
constexpr int kTileShift = 10, kTile = 1 << kTileShift, kTileThreads = kTile / 4;   // 1024 positions per CTA

// voxel key of sub_sample_frame: static_cast<short>(raw / size) per axis (ct_icp.cpp:70-72)
__device__ __forceinline__ unsigned long long short_voxel_key(const RawPoint &p, double voxel_size) {
    // int(p / size) from the reciprocal (division only next to an integer quotient: voxel_coord_rcp, device_map.cuh)
    const double inv = 1.0 / voxel_size;
    const short x = (short) voxel_coord_rcp(p.x, voxel_size, inv);
    const short y = (short) voxel_coord_rcp(p.y, voxel_size, inv);
    const short z = (short) voxel_coord_rcp(p.z, voxel_size, inv);
    return ((unsigned long long) (unsigned short) x << 32) | ((unsigned long long) (unsigned short) y << 16) |
           (unsigned long long) (unsigned short) z;
}

// find-or-insert `key` in the scratch hash grid (linear probing); returns its slot
__device__ __forceinline__ uint32_t grid_find_or_insert(unsigned long long *keys, uint32_t cap_mask, unsigned long long key) {
    uint32_t h = hash_key(key) & cap_mask;
    while (true) {
        unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(&keys[h]);
        if (k == kGridEmpty) k = atomicCAS(&keys[h], kGridEmpty, key);
        if (k == kGridEmpty || k == key) return h;
        h = (h + 1) & cap_mask;
    }
}
// claim: every point bids (priority, index) for its voxel. Consecutive scan points share few voxels (a median of 3 keys
// per warp on a 64-beam scan, up to ~1000 points in one voxel next to the sensor), so the lanes of a warp that hold the
// same key first agree on their smallest priority and only that lane (the group's leader) probes and bids: one atomic per
// (warp, voxel) instead of one per point, and no queue of atomics at a hot voxel's word. Priorities are unique, so the
// bid is the same one the point-by-point claim would have won with. slot_of[i] = the slot for a leader, -1 otherwise
// (a non-leader can never be its voxel's winner).
// All lanes of a warp run the same number of iterations (the loop walks whole warps), as the warp collectives require.
__device__ __forceinline__ void grid_claim_dev(const float4 *pts, const float4 *lo, int n, double voxel_size, int use_perm,
                                               uint64_t seed, uint64_t counter, unsigned long long *keys,
                                               unsigned long long *vals, uint32_t cap_mask, int *__restrict__ slot_of) {
    const Perm perm = perm_make(seed, counter, (uint32_t) max(n, 1));
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, num_warps = (gridDim.x * blockDim.x) >> 5;
    for (int base = warp * 32; base < n; base += num_warps * 32) {
        const int i = base + lane;
        const unsigned active = __ballot_sync(0xffffffffu, i < n);
        if (i >= n) continue;
        const unsigned long long key = short_voxel_key(load_raw(pts, lo, i), voxel_size);
        const uint32_t prio = use_perm ? perm_apply(perm, (uint32_t) i) : (uint32_t) i;
        const unsigned peers = __match_any_sync(active, key);
        const uint32_t best = __reduce_min_sync(peers, prio);
        const bool leader = prio == best;
        uint32_t h = 0;
        if (leader) {
            h = grid_find_or_insert(keys, cap_mask, key);
            atomicMin(&vals[h], ((unsigned long long) prio << 32) | (unsigned) i);
        }
        slot_of[i] = leader ? (int) h : -1;
    }
}
__global__ void k_grid_claim(const float4 *__restrict__ pts, const float4 *__restrict__ lo, const int *__restrict__ d_n,
                             double voxel_size, int use_perm, uint64_t seed, uint64_t counter, unsigned long long *keys,
                             unsigned long long *vals, uint32_t cap_mask, int *__restrict__ slot_of) {
    grid_claim_dev(pts, lo, *d_n, voxel_size, use_perm, seed, counter, keys, vals, cap_mask, slot_of);
}
// mark: winners raise a flag at their position in the permuted order (slot_of < 0: a point that did not bid)
__device__ __forceinline__ void grid_mark_dev(int n, int use_perm, uint64_t seed, uint64_t counter,
                                              const unsigned long long *vals, const int *slot_of, uint32_t *__restrict__ flags,
                                              uint32_t *__restrict__ src, uint32_t *__restrict__ tile_count) {
    const Perm perm = perm_make(seed, counter, (uint32_t) max(n, 1));
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int slot = slot_of[i];
        if (slot < 0) continue;   // not its warp group's bidder
        const uint32_t prio = use_perm ? perm_apply(perm, (uint32_t) i) : (uint32_t) i;
        const unsigned long long mine = ((unsigned long long) prio << 32) | (unsigned) i;
        if (vals[slot] == mine) {
            flags[prio] = 1u;
            src[prio] = (uint32_t) i;
            atomicAdd(&tile_count[prio >> kTileShift], 1u);   // integer atomics: order-independent result
        }
    }
}
__global__ void k_grid_mark(const int *__restrict__ d_n, int use_perm, uint64_t seed, uint64_t counter,
                            const unsigned long long *__restrict__ vals, const int *__restrict__ slot_of,
                            uint32_t *__restrict__ flags, uint32_t *__restrict__ src,
                            uint32_t *__restrict__ tile_count) {
    grid_mark_dev(*d_n, use_perm, seed, counter, vals, slot_of, flags, src, tile_count);
}
// emit: compact the winners in permuted order and (optionally) scatter them through a second permutation (the
// second shuffle). One CTA per tile of 1024 positions: the exclusive prefix of a position is
//   Σ tile_count[tiles before] (every CTA re-adds those <= 512 counters) + a CTA-local scan of the tile's flags,
// which replaces a serial single-CTA scan over all positions (64 us for 130k points) by a fully parallel pass.
struct EmitScratch {
    uint32_t red[2][kTileThreads / 32];
    uint32_t warp[kTileThreads / 32];
    uint32_t before, total;
};
// capacity of the hash grid of a selection over n points (load <= 0.5)
__device__ __forceinline__ uint32_t grid_cap_for(uint32_t n) {
    uint32_t cap = 1024;
    while (cap < 2 * n) cap <<= 1;
    return cap;
}
// The claim of a second, unpermuted selection over the emitted points (grid_sampling of the sub-sampled frame), issued
// while they are emitted: its priority is the output position, which the emit already holds together with the point.
// `grid` (keys | vals of grid_cap_for(total) words each) must be clean; `tile` (tile counters | flags of the second
// selection) is cleared here for total positions.
struct NextClaim {
    double voxel_size;
    unsigned long long *grid;
    int *slot_of;      // indexed by output position
    uint32_t *tile;
};
// all threads of a CTA of kTileThreads threads; returns the number of winners (identical in every CTA)
__device__ __forceinline__ uint32_t grid_emit_dev(const float4 *pts, const float4 *lo, const uint32_t *in_src_index, int n,
                                                  const uint32_t *flags, const uint32_t *src, const uint32_t *tile_count,
                                                  int use_perm2, uint64_t seed, uint64_t counter2, int override_alpha,
                                                  float alpha_value, float4 *__restrict__ out, float4 *__restrict__ out_lo,
                                                  uint32_t *__restrict__ out_src_index, int *__restrict__ d_total,
                                                  EmitScratch &sc, const NextClaim *next = nullptr) {
    uint32_t (&s_red)[2][kTileThreads / 32] = sc.red;
    uint32_t (&s_warp)[kTileThreads / 32] = sc.warp;
    uint32_t &s_before = sc.before, &s_total = sc.total;
    const int num_tiles = (n + kTile - 1) >> kTileShift;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    // grand total (domain of the second permutation) — identical in every CTA
    uint32_t tot = 0;
    for (int t = tid; t < num_tiles; t += kTileThreads) tot += tile_count[t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if (lane == 0) s_red[1][w] = tot;
    __syncthreads();
    if (tid == 0) {
        uint32_t b = 0;
        for (int i = 0; i < kTileThreads / 32; ++i) b += s_red[1][i];
        s_total = b;
    }
    __syncthreads();
    const uint32_t total = s_total;
    if (blockIdx.x == 0 && tid == 0) *d_total = (int) total;
    const Perm perm2 = perm_make(seed, counter2, max(total, 1u));
    uint32_t next_mask = 0;
    if (next) {
        next_mask = grid_cap_for(total) - 1;
        const size_t words = kMaxTiles + (size_t) total;
        for (size_t t = (size_t) blockIdx.x * blockDim.x + tid; t < words; t += (size_t) gridDim.x * blockDim.x) next->tile[t] = 0u;
    }

    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        uint32_t before = 0;
        for (int t = tid; t < tile; t += kTileThreads) before += tile_count[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
        __syncthreads();   // s_red / s_warp reuse across tiles
        if (lane == 0) s_red[0][w] = before;
        // CTA-local exclusive scan of the tile's flags: 4 consecutive positions per thread
        const int p0 = (tile << kTileShift) + tid * 4;
        uint32_t v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = (p0 + k < n) ? flags[p0 + k] : 0u;
        const uint32_t tsum = v[0] + v[1] + v[2] + v[3];
        uint32_t incl = tsum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) s_warp[w] = incl;
        __syncthreads();
        if (tid == 0) {
            uint32_t b = 0;
            for (int i = 0; i < kTileThreads / 32; ++i) b += s_red[0][i];
            s_before = b;
            uint32_t run = 0;
            for (int i = 0; i < kTileThreads / 32; ++i) {
                const uint32_t c = s_warp[i];
                s_warp[i] = run;
                run += c;
            }
        }
        __syncthreads();
        uint32_t excl = s_before + s_warp[w] + (incl - tsum);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (v[k]) {
                const uint32_t dst = (use_perm2 && total > 1) ? perm_apply(perm2, excl) : excl;
                const uint32_t i = src[p0 + k];
                float4 val = pts[i];
                if (override_alpha) val.w = alpha_value;
                out[dst] = val;
                // (the point as load_raw(out, out_lo, dst) reads it back)
                RawPoint r{f32_to_f64(val.x), f32_to_f64(val.y), f32_to_f64(val.z), 0.0};
                if (out_lo) {
                    float4 l = lo ? lo[i] : make_float4(0.f, 0.f, 0.f, 0.f);
                    if (override_alpha) l.w = 0.f;
                    out_lo[dst] = l;
                    r.x += (double) l.x; r.y += (double) l.y; r.z += (double) l.z;
                }
                out_src_index[dst] = in_src_index ? in_src_index[i] : i;
                if (next) {
                    const uint32_t h = grid_find_or_insert(next->grid, next_mask, short_voxel_key(r, next->voxel_size));
                    atomicMin(&next->grid[next_mask + 1 + h], ((unsigned long long) dst << 32) | dst);
                    next->slot_of[dst] = (int) h;
                }
            }
            excl += v[k];
        }
    }
    return total;
}
__global__ void __launch_bounds__(kTileThreads)
k_grid_emit(const float4 *__restrict__ pts, const float4 *__restrict__ lo, const uint32_t *__restrict__ in_src_index,
            const int *__restrict__ d_n, const uint32_t *__restrict__ flags, const uint32_t *__restrict__ src,
            const uint32_t *__restrict__ tile_count, int use_perm2, uint64_t seed, uint64_t counter2,
            int override_alpha, float alpha_value, float4 *__restrict__ out, float4 *__restrict__ out_lo,
            uint32_t *__restrict__ out_src_index, int *__restrict__ d_total) {
    __shared__ EmitScratch sc;
    grid_emit_dev(pts, lo, in_src_index, *d_n, flags, src, tile_count, use_perm2, seed, counter2, override_alpha, alpha_value,
                  out, out_lo, out_src_index, d_total, sc);
}

// ---- both grid selections of a frame (sub_sample_frame N -> F, grid_sampling F -> K) in ONE cooperative launch: five
// phases separated by four grid barriers (claim 1 | mark 1 | emit 1 + claim 2 | mark 2 | emit 2) instead of six kernels +
// four memsets. (Each of those kernels lasts 4-11 us for work worth about one: launch ramp, tail, and the dependency on its
// predecessor; 46 us of a 310 us step in round 1. Each grid barrier costs about 2 us.)
struct FusedSampleArgs {
    const float4 *raw;
    const float4 *raw_lo;              // residual plane of the scan (nullptr: float32-representable)
    float4 *frame_lo, *kp_lo;          // residual planes of the two selections (written iff raw_lo)
    int n;                             // N (also written to counts[0] for later kernels)
    int *counts;                       // [0] = N, [1] = F out, [2] = K out
    double voxel1, voxel2;
    uint64_t seed, c1, c2;
    int override_alpha;
    float alpha_value;
    unsigned long long *grid;          // keys | vals, 2 * cap1 words
    unsigned long long *grid2;         // selection 2's keys | vals: claimed into while selection 1 emits, so always clean
    uint32_t cap1;
    int *slot_of;
    uint32_t *tile1, *flags1, *src1;   // selection 1 (tile counters and flags adjacent)
    uint32_t *tile2, *flags2, *src2;   // selection 2
    float4 *frame, *keypoints;
    uint32_t *frame_src, *kp_src;
    // The hash grid and the flag / tile-counter arrays of selection 1 are left CLEAN for the next frame by the last phase of
    // this launch (they are idle there), so the next launch starts at the claim phase: one grid barrier and a 4.5 MB clear
    // less on the critical path of every frame. pre_cleared: the previous launch did that for at least this frame's sizes.
    int pre_cleared;
    uint32_t clear_words;              // words of tile1 | flags1 to leave clean (this frame's count with head-room)
};
__global__ void __launch_bounds__(kTileThreads)
k_sample_fused(FusedSampleArgs a) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ EmitScratch sc;
    const size_t gtid = (size_t) blockIdx.x * blockDim.x + threadIdx.x, gsize = (size_t) gridDim.x * blockDim.x;
    const int n = a.n;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.counts[0] = n;
    // phase 0: clear the hash grid and the flag / tile-counter arrays of selection 1 (unless the previous launch left them clean)
    if (!a.pre_cleared) {
        for (size_t i = gtid; i < 2 * (size_t) a.cap1; i += gsize) a.grid[i] = kGridEmpty;
        for (size_t i = gtid; i < 2 * (size_t) a.cap1; i += gsize) a.grid2[i] = kGridEmpty;   // (F <= N: cap2 <= cap1)
        for (size_t i = gtid; i < kMaxTiles + (size_t) n; i += gsize) a.tile1[i] = 0u;   // flags1 = tile1 + kMaxTiles
        grid.sync();
    }
    grid_claim_dev(a.raw, a.raw_lo, n, a.voxel1, 1, a.seed, a.c1, a.grid, a.grid + a.cap1, a.cap1 - 1, a.slot_of);
    grid.sync();
    grid_mark_dev(n, 1, a.seed, a.c1, a.grid + a.cap1, a.slot_of, a.flags1, a.src1, a.tile1);
    grid.sync();
    float4 *frame_lo = a.raw_lo ? a.frame_lo : nullptr, *kp_lo = a.raw_lo ? a.kp_lo : nullptr;
    // emit of selection 1 + claim of selection 2 (priority = frame index, grid2) + clear of selection 2's flags; slot_of is
    // free again (last read by mark 1, a barrier ago)
    const NextClaim claim2{a.voxel2, a.grid2, a.slot_of, a.tile2};
    const uint32_t F = grid_emit_dev(a.raw, a.raw_lo, nullptr, n, a.flags1, a.src1, a.tile1, 1, a.seed, a.c2, a.override_alpha,
                                     a.alpha_value, a.frame, frame_lo, a.frame_src, a.counts + 1, sc, &claim2);
    const uint32_t cap2 = grid_cap_for(F);
    grid.sync();
    grid_mark_dev((int) F, 0, 0, 0, a.grid2 + cap2, a.slot_of, a.flags2, a.src2, a.tile2);
    grid.sync();
    grid_emit_dev(a.frame, frame_lo, a.frame_src, (int) F, a.flags2, a.src2, a.tile2, 0, 0, 0, 0, 0.f, a.keypoints, kp_lo,
                  a.kp_src, a.counts + 2, sc);
    // grid 1 (last read by mark 1), grid 2 (last read by mark 2) and selection 1's arrays (last read by its emit): clean for
    // the next frame
    if (a.clear_words) {
        for (size_t i = gtid; i < 2 * (size_t) a.cap1; i += gsize) a.grid[i] = kGridEmpty;
        for (size_t i = gtid; i < 2 * (size_t) cap2; i += gsize) a.grid2[i] = kGridEmpty;
        for (size_t i = gtid; i < (size_t) a.clear_words; i += gsize) a.tile1[i] = 0u;
    }
}
// ---- adaptive (distance-banded) grid sampling: AdaptiveSamplePointsInGrid, include/ct_icp/algorithm/sampling.h:55-110
struct AdaptiveBands {
    int num_bands;
    double distance[CTICP_MAX_ADAPTIVE_BANDS];
    double voxel_size[CTICP_MAX_ADAPTIVE_BANDS];
};
__device__ __forceinline__ int adaptive_band(const AdaptiveBands &B, const RawPoint &p, unsigned long long *key_out) {
    const double x = p.x, y = p.y, z = p.z;
    const double dist = sqrt(x * x + y * y + z * z);
    int lw = 0;   // std::lower_bound with comp(elem, v) = elem.first < v (:69-74)
    while (lw < B.num_bands && B.distance[lw] < dist) ++lw;
    if (!(dist >= B.distance[0] && dist < B.distance[B.num_bands - 1])) return -1;
    const int band = lw - 1;
    if (band < 0) return -1;
    const double vs = B.voxel_size[band];
    const int vx = voxel_coord(x, vs), vy = voxel_coord(y, vs), vz = voxel_coord(z, vs);   // slam::Voxel::Coordinates
    const int bias = 1 << 19;
    *key_out = ((unsigned long long) (band + 1) << 60) | ((unsigned long long) (unsigned) ((vx + bias) & 0xFFFFF) << 40) |
               ((unsigned long long) (unsigned) ((vy + bias) & 0xFFFFF) << 20) | (unsigned long long) (unsigned) ((vz + bias) & 0xFFFFF);
    return band;
}
__global__ void k_adaptive_claim(const float4 *__restrict__ pts, const float4 *__restrict__ lo, const int *__restrict__ d_n, AdaptiveBands B,
                                 unsigned long long *keys, unsigned long long *vals, uint32_t cap_mask,
                                 int *__restrict__ slot_of, int *__restrict__ d_positions) {
    const int n = *d_n;
    if (blockIdx.x == 0 && threadIdx.x == 0) *d_positions = n * B.num_bands;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned long long key;
        const int band = adaptive_band(B, load_raw(pts, lo, i), &key);
        if (band < 0) {
            slot_of[i] = -1;
            continue;
        }
        uint32_t h = hash_key(key) & cap_mask;
        while (true) {
            unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(&keys[h]);
            if (k == kGridEmpty) k = atomicCAS(&keys[h], kGridEmpty, key);
            if (k == kGridEmpty || k == key) break;
            h = (h + 1) & cap_mask;
        }
        atomicMin(&vals[h], (unsigned long long) (unsigned) i);   // first seen = smallest index (:79-84)
        slot_of[i] = (int) h;
    }
}
__global__ void k_adaptive_mark(const float4 *__restrict__ pts, const float4 *__restrict__ lo, const int *__restrict__ d_n, AdaptiveBands B,
                                const unsigned long long *__restrict__ vals, const int *__restrict__ slot_of,
                                uint32_t *__restrict__ flags, uint32_t *__restrict__ src,
                                uint32_t *__restrict__ tile_count) {
    const int n = *d_n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int slot = slot_of[i];
        if (slot < 0 || vals[slot] != (unsigned long long) (unsigned) i) continue;
        unsigned long long key;
        const int band = adaptive_band(B, load_raw(pts, lo, i), &key);
        const uint32_t pos = (uint32_t) band * (uint32_t) n + (uint32_t) i;   // band-major, then first appearance
        flags[pos] = 1u;
        src[pos] = (uint32_t) i;
        atomicAdd(&tile_count[pos >> kTileShift], 1u);
    }
}

// keypoints = frame (sampling NONE, odometry.cpp:546)
__global__ void k_copy_points(const float4 *__restrict__ in, const float4 *__restrict__ in_lo, const uint32_t *__restrict__ in_src,
                              const int *__restrict__ d_n, float4 *__restrict__ out, float4 *__restrict__ out_lo,
                              uint32_t *__restrict__ out_src, int *__restrict__ d_n_out) {
    const int n = *d_n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        out[i] = in[i];
        if (in_lo) out_lo[i] = in_lo[i];
        out_src[i] = in_src[i];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *d_n_out = n;
}
// max_num_keypoints: shuffle + resize (odometry.cpp:549-552) when *d_n > max_n
__global__ void k_truncate_shuffle(const float4 *__restrict__ in, const float4 *__restrict__ in_lo, const uint32_t *__restrict__ in_src,
                                   const int *__restrict__ d_n, int max_n, uint64_t seed, uint64_t counter,
                                   float4 *__restrict__ out, float4 *__restrict__ out_lo, uint32_t *__restrict__ out_src) {
    const int n = *d_n;
    const bool active = n > max_n;
    const Perm perm = perm_make(seed, counter, (uint32_t) max(n, 1));
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t d = active ? perm_apply(perm, (uint32_t) i) : (uint32_t) i;
        if (!active || (int) d < max_n) {
            out[d] = in[i];
            if (in_lo) out_lo[d] = in_lo[i];
            out_src[d] = in_src[i];
        }
    }
}
__global__ void k_clamp_count(int *d_n, int max_n) {
    if (*d_n > max_n) *d_n = max_n;
}
// world = ContinuousTransform(raw, begin, end, alpha) for every point (odometry.cpp:463-486)
__global__ void k_transform_points(const float4 *__restrict__ pts, const float4 *__restrict__ lo, const int *__restrict__ d_n,
                                   Q4 qb, V3 tb, Q4 qe, V3 te, SlerpConsts sc, double *__restrict__ world) {
    const int n = *d_n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const RawPoint p = load_raw(pts, lo, i);
        // acos / 1/sin(theta) of the pose pair are hoisted (sc): two sin per point instead of acos + three sin
        const V3 w = ct_transform_c(qb, tb, qe, te, p.alpha, V3{p.x, p.y, p.z}, sc);
        world[3 * i] = w.x; world[3 * i + 1] = w.y; world[3 * i + 2] = w.z;
    }
}

// DistortFrame (odometry.cpp:161-168): raw <- end^-1 * (Interpolate(begin, end, t) * raw), in place (alpha kept)
__global__ void k_distort_frame(float4 *__restrict__ pts, float4 *__restrict__ lo, int lo_valid,
                                const int *__restrict__ d_n, Q4 qb, V3 tb, Q4 qe, V3 te, SlerpConsts sc) {
    const int n = *d_n;
    const Q4 qi = qinverse(qe);
    const V3 ti = (-1.0) * qrot(qnormalized(qi), te);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const RawPoint p = load_raw(pts, lo_valid ? lo : nullptr, i);
        const V3 w = ct_transform_c(qb, tb, qe, te, p.alpha, V3{p.x, p.y, p.z}, sc);
        const V3 r = qrot(qnormalized(qi), w) + ti;
        store_raw(pts, lo, i, r.x, r.y, r.z, p.alpha);   // the distorted point is not float32-representable: hi + lo
    }
}

// ---------------------------------------------------------------------------------------------------------------
static uint32_t NextPow2(uint64_t v) {
    uint64_t p = 1;
    while (p < v) p <<= 1;
    return (uint32_t) p;
}

FramePipeline::FramePipeline(size_t max_points, cudaStream_t stream) : stream_(stream), max_points_(max_points) {
    const size_t n = max_points_;
    if (const char *e = getenv("CTICP_SAMPLE_PRECLEAR")) preclear_ = atoi(e) != 0;
    grid_cap_ = std::max<uint32_t>(NextPow2(2 * n), 1024);
    CT_CUDA_CHECK(cudaMallocHost(&h_stage_, sizeof(float4) * n));
    CT_CUDA_CHECK(cudaMallocHost(&h_counts_, sizeof(int) * 8));
    CT_CUDA_CHECK(cudaMalloc(&d_raw_, sizeof(float4) * n));
    raw_ = d_raw_;
    CT_CUDA_CHECK(cudaMalloc(&d_frame_, sizeof(float4) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_keypoints_, sizeof(float4) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_tmp_points_, sizeof(float4) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_frame_src_, sizeof(uint32_t) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_kp_src_, sizeof(uint32_t) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_tmp_src_, sizeof(uint32_t) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_grid_, sizeof(unsigned long long) * 2 * (size_t) grid_cap_));
    CT_CUDA_CHECK(cudaMalloc(&d_slot_of_, sizeof(int) * n));
    if ((n + kTile - 1) / kTile > kMaxTiles) throw std::invalid_argument("max_points_per_frame too large");
    CT_CUDA_CHECK(cudaMalloc(&d_tile_count_, sizeof(uint32_t) * (kMaxTiles + n)));
    d_flags_ = d_tile_count_ + kMaxTiles;
    CT_CUDA_CHECK(cudaMalloc(&d_src_, sizeof(uint32_t) * n));
    CT_CUDA_CHECK(cudaMalloc(&d_counts_, sizeof(int) * 8));
    CT_CUDA_CHECK(cudaMalloc(&d_frame_world_, sizeof(double) * 3 * n));
    CT_CUDA_CHECK(cudaMemsetAsync(d_counts_, 0, sizeof(int) * 8, stream_));
    memset(h_counts_, 0, sizeof(int) * 8);
}
FramePipeline::~FramePipeline() {
    cudaFreeHost(h_stage_); cudaFreeHost(h_counts_);
    cudaFree(d_raw_); cudaFree(d_frame_); cudaFree(d_keypoints_); cudaFree(d_tmp_points_);
    cudaFreeHost(h_stage_lo_);
    cudaFree(d_raw_lo_); cudaFree(d_frame_lo_); cudaFree(d_kp_lo_); cudaFree(d_tmp_lo_);
    cudaFree(d_frame_src_); cudaFree(d_kp_src_); cudaFree(d_tmp_src_);
    cudaFree(d_grid_); cudaFree(d_slot_of_); cudaFree(d_tile_count_); cudaFree(d_src_);
    cudaFree(d_counts_); cudaFree(d_frame_world_); cudaFree(d_all_world_); cudaFree(d_adaptive_);
    cudaFree(d_tile2_); cudaFree(d_src2_); cudaFree(d_grid2_);
}

int FramePipeline::Blocks(size_t n) const { return (int) std::max<size_t>(1, std::min<size_t>((n + 255) / 256, 148 * 8)); }

void FramePipeline::EnsureLo() {
    if (d_raw_lo_) return;
    CT_CUDA_CHECK(cudaMallocHost(&h_stage_lo_, sizeof(float4) * max_points_));
    CT_CUDA_CHECK(cudaMalloc(&d_raw_lo_, sizeof(float4) * max_points_));
    CT_CUDA_CHECK(cudaMalloc(&d_frame_lo_, sizeof(float4) * max_points_));
    CT_CUDA_CHECK(cudaMalloc(&d_kp_lo_, sizeof(float4) * max_points_));
    CT_CUDA_CHECK(cudaMalloc(&d_tmp_lo_, sizeof(float4) * max_points_));
}

void FramePipeline::UploadLo(size_t n) {
    EnsureLo();
    CT_CUDA_CHECK(cudaMemcpyAsync(d_raw_lo_, h_stage_lo_, sizeof(float4) * n, cudaMemcpyHostToDevice, stream_));
    raw_lo_ = true;
    raw_lo_view_ = d_raw_lo_;
    h2d_bytes_ += sizeof(float4) * n;
}

void FramePipeline::Upload(size_t n) {
    if (n > max_points_) throw CapacityError("scan has more points than max_points_per_frame");
    raw_lo_ = frame_lo_ = distorted_ = count_n_pending_ = false;
    raw_ = d_raw_;
    n_ = n;
    h_counts_[0] = (int) n;
    CT_CUDA_CHECK(cudaMemcpyAsync(d_raw_, h_stage_, sizeof(float4) * n, cudaMemcpyHostToDevice, stream_));
    CT_CUDA_CHECK(cudaMemcpyAsync(d_counts_, h_counts_, sizeof(int), cudaMemcpyHostToDevice, stream_));
    h2d_bytes_ = sizeof(float4) * n + sizeof(int);
}

void FramePipeline::UploadBegin(size_t n) {
    if (n > max_points_) throw CapacityError("scan has more points than max_points_per_frame");
    raw_lo_ = frame_lo_ = distorted_ = count_n_pending_ = false;
    raw_ = d_raw_;
    n_ = n;
    h_counts_[0] = (int) n;
    CT_CUDA_CHECK(cudaMemcpyAsync(d_counts_, h_counts_, sizeof(int), cudaMemcpyHostToDevice, stream_));
    h2d_bytes_ = sizeof(float4) * n + sizeof(int);
}
void FramePipeline::UploadRange(size_t begin, size_t end) {
    if (end <= begin) return;
    CT_CUDA_CHECK(cudaMemcpyAsync(d_raw_ + begin, h_stage_ + begin, sizeof(float4) * (end - begin), cudaMemcpyHostToDevice, stream_));
}

void FramePipeline::UploadFromDevice(const float4 *d_src, const float4 *d_src_lo, size_t n) {
    if (n > max_points_) throw CapacityError("scan has more points than max_points_per_frame");
    frame_lo_ = distorted_ = false;
    n_ = n;
    raw_ = d_src;
    raw_lo_view_ = d_src_lo;
    raw_lo_ = d_src_lo != nullptr;
    count_n_pending_ = true;
    h2d_bytes_ = 0;
}

void FramePipeline::DetachRaw() {
    if (raw_ == d_raw_) return;
    CT_CUDA_CHECK(cudaMemcpyAsync(d_raw_, raw_, sizeof(float4) * n_, cudaMemcpyDeviceToDevice, stream_));
    if (raw_lo_) {
        EnsureLo();
        CT_CUDA_CHECK(cudaMemcpyAsync(d_raw_lo_, raw_lo_view_, sizeof(float4) * n_, cudaMemcpyDeviceToDevice, stream_));
    }
    raw_ = d_raw_;
    raw_lo_view_ = d_raw_lo_;
}

void FramePipeline::EnsureCountN() {
    if (!count_n_pending_) return;
    h_counts_[0] = (int) n_;
    CT_CUDA_CHECK(cudaMemcpyAsync(d_counts_, h_counts_, sizeof(int), cudaMemcpyHostToDevice, stream_));
    h2d_bytes_ += sizeof(int);
    count_n_pending_ = false;
}

void FramePipeline::GridSelect(const float4 *in, const float4 *in_lo, const uint32_t *in_src, const int *d_n_in,
                               size_t n_upper, double voxel_size, int use_perm1, uint64_t seed, uint64_t c1,
                               int use_perm2, uint64_t c2, int override_alpha, float alpha_value, float4 *out,
                               float4 *out_lo, uint32_t *out_src, int *d_n_out) {
    if (!in_lo) out_lo = nullptr;
    clean_cap_ = 0;   // (this selection dirties what the fused sampler may have left clean)
    clean_words_ = 0;
    // scratch hash grid: only the prefix that can be touched is cleared; keys and vals are adjacent → one memset
    const uint32_t cap = std::max<uint32_t>(NextPow2(2 * n_upper), 1024);
    unsigned long long *keys = d_grid_, *vals = d_grid_ + cap;
    CT_CUDA_CHECK(cudaMemsetAsync(keys, 0xFF, sizeof(unsigned long long) * 2 * (size_t) cap, stream_));
    // flags and tile counters are adjacent → one memset
    const size_t num_tiles = (n_upper + kTile - 1) / kTile;
    CT_CUDA_CHECK(cudaMemsetAsync(d_tile_count_, 0, sizeof(uint32_t) * (kMaxTiles + n_upper), stream_));
    const int blocks = Blocks(n_upper);
    k_grid_claim<<<blocks, 256, 0, stream_>>>(in, in_lo, d_n_in, voxel_size, use_perm1, seed, c1, keys, vals, cap - 1, d_slot_of_);
    k_grid_mark<<<blocks, 256, 0, stream_>>>(d_n_in, use_perm1, seed, c1, vals, d_slot_of_, d_flags_, d_src_, d_tile_count_);
    k_grid_emit<<<(int) std::max<size_t>(1, num_tiles), kTileThreads, 0, stream_>>>(
        in, in_lo, in_src, d_n_in, d_flags_, d_src_, d_tile_count_, use_perm2, seed, c2, override_alpha, alpha_value, out,
        out_lo, out_src, d_n_out);
    launches_ += 3;
    CT_CUDA_CHECK(cudaGetLastError());
}

void FramePipeline::AdaptiveSelect(const cticp_adaptive_options &o, const float4 *in, const float4 *in_lo,
                                   const uint32_t *in_src, const int *d_n_in, size_t n_upper, float4 *out,
                                   float4 *out_lo, uint32_t *out_src, int *d_n_out) {
    if (!in_lo) out_lo = nullptr;
    clean_cap_ = 0;
    clean_words_ = 0;
    if (o.num_points_per_voxel != 1) throw std::invalid_argument("adaptive sampling: only num_points_per_voxel == 1 is built");
    if (o.num_bands < 2 || o.num_bands > CTICP_MAX_ADAPTIVE_BANDS) throw std::invalid_argument("adaptive sampling: num_bands");
    AdaptiveBands B;
    B.num_bands = o.num_bands;
    for (int i = 0; i < CTICP_MAX_ADAPTIVE_BANDS; ++i) {
        B.distance[i] = o.distance[i];
        B.voxel_size[i] = o.voxel_size[i];
    }
    const size_t positions = n_upper * (size_t) o.num_bands;
    if ((positions + kTile - 1) / kTile > kMaxTiles) throw CapacityError("adaptive sampling: scan too large");
    if (positions > adaptive_capacity_) {
        CT_CUDA_CHECK(cudaStreamSynchronize(stream_));
        cudaFree(d_adaptive_);
        CT_CUDA_CHECK(cudaMalloc(&d_adaptive_, sizeof(uint32_t) * (kMaxTiles + 2 * positions)));
        adaptive_capacity_ = positions;
    }
    uint32_t *tile_count = d_adaptive_, *flags = d_adaptive_ + kMaxTiles, *src = flags + positions;
    const uint32_t cap = std::max<uint32_t>(NextPow2(2 * n_upper), 1024);
    unsigned long long *keys = d_grid_, *vals = d_grid_ + cap;
    CT_CUDA_CHECK(cudaMemsetAsync(keys, 0xFF, sizeof(unsigned long long) * 2 * (size_t) cap, stream_));
    CT_CUDA_CHECK(cudaMemsetAsync(tile_count, 0, sizeof(uint32_t) * (kMaxTiles + positions), stream_));
    const int blocks = Blocks(n_upper);
    int *d_positions = d_counts_ + 3;
    k_adaptive_claim<<<blocks, 256, 0, stream_>>>(in, in_lo, d_n_in, B, keys, vals, cap - 1, d_slot_of_, d_positions);
    k_adaptive_mark<<<blocks, 256, 0, stream_>>>(in, in_lo, d_n_in, B, vals, d_slot_of_, flags, src, tile_count);
    const size_t num_tiles = (positions + kTile - 1) / kTile;
    k_grid_emit<<<(int) std::min<size_t>(std::max<size_t>(1, num_tiles), 1184), kTileThreads, 0, stream_>>>(
        in, in_lo, in_src, d_positions, flags, src, tile_count, 0, 0, 0, 0, 0.f, out, out_lo, out_src, d_n_out);
    launches_ += 3;
    if (o.max_num_points > 0) {   // `indices.size() > kMaxNumPoints` lets max + 1 through (:96-105)
        k_clamp_count<<<1, 1, 0, stream_>>>(d_n_out, o.max_num_points + 1);
        launches_ += 1;
    }
    CT_CUDA_CHECK(cudaGetLastError());
}

// SubSampleFrame + SampleKeypoints(GRID) of one frame in a single cooperative launch (k_sample_fused). The keypoint
// sampling's parameters must be known when the frame arrives: true for the first registration attempt of a frame.
void FramePipeline::SampleFused(double voxel_size, double sample_voxel_size, uint64_t seed, uint64_t counter1,
                                uint64_t counter2, bool override_alpha, float alpha_value) {
    if (!d_tile2_) {
        CT_CUDA_CHECK(cudaMalloc(&d_tile2_, sizeof(uint32_t) * (kMaxTiles + max_points_)));
        CT_CUDA_CHECK(cudaMalloc(&d_src2_, sizeof(uint32_t) * max_points_));
        CT_CUDA_CHECK(cudaMalloc(&d_grid2_, sizeof(unsigned long long) * 2 * (size_t) grid_cap_));
        CT_CUDA_CHECK(cudaMemsetAsync(d_grid2_, 0xFF, sizeof(unsigned long long) * 2 * (size_t) grid_cap_, stream_));
        int per_sm = 0;
        CT_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sample_fused, kTileThreads, 0));
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        int want = 4;   // CTAs per SM: more hide the latency of the probes, fewer make the grid barriers cheaper (A/B knob)
        if (const char *e = getenv("CTICP_SAMPLE_CTAS_PER_SM")) want = std::max(1, atoi(e));
        fused_grid_ = std::max(1, std::min(per_sm, want) * sms);
    }
    FusedSampleArgs a;
    a.raw = raw_;
    a.raw_lo = d_raw_lo();
    a.n = (int) n_;
    count_n_pending_ = false;   // (the launch writes counts[0])
    a.frame_lo = d_frame_lo_; a.kp_lo = d_kp_lo_;
    frame_lo_ = raw_lo_;
    a.counts = d_counts_;
    a.voxel1 = voxel_size;
    a.voxel2 = sample_voxel_size;
    a.seed = seed; a.c1 = counter1; a.c2 = counter2;
    a.override_alpha = override_alpha ? 1 : 0;
    a.alpha_value = alpha_value;
    a.grid = d_grid_;
    a.grid2 = d_grid2_;
    a.cap1 = std::max<uint32_t>(NextPow2(2 * n_), 1024);
    a.pre_cleared = (preclear_ && clean_cap_ >= a.cap1 && clean_words_ >= kMaxTiles + n_) ? 1 : 0;
    a.clear_words = preclear_ ? (uint32_t) (kMaxTiles + std::min(max_points_, n_ + n_ / 8 + 1024)) : 0u;
    clean_cap_ = preclear_ ? a.cap1 : 0;        // what this launch leaves behind
    clean_words_ = a.clear_words;
    a.slot_of = d_slot_of_;
    a.tile1 = d_tile_count_; a.flags1 = d_flags_; a.src1 = d_src_;
    a.tile2 = d_tile2_; a.flags2 = d_tile2_ + kMaxTiles; a.src2 = d_src2_;
    a.frame = d_frame_; a.keypoints = d_keypoints_;
    a.frame_src = d_frame_src_; a.kp_src = d_kp_src_;
    void *args[] = {&a};
    CT_CUDA_CHECK(cudaLaunchCooperativeKernel((void *) k_sample_fused, dim3(fused_grid_), dim3(kTileThreads), args, 0, stream_));
    launches_ += 1;
}

void FramePipeline::SubSampleFrame(double voxel_size, uint64_t seed, uint64_t counter1, uint64_t counter2,
                                   bool override_alpha, float alpha_value) {
    EnsureCountN();
    GridSelect(raw_, d_raw_lo(), nullptr, d_counts_ + 0, n_, voxel_size, 1, seed, counter1, 1, counter2,
               override_alpha ? 1 : 0, alpha_value, d_frame_, d_frame_lo_, d_frame_src_, d_counts_ + 1);
    frame_lo_ = raw_lo_;
}

void FramePipeline::SampleKeypoints(int sampling, double sample_voxel_size, int max_num_keypoints, uint64_t seed,
                                    uint64_t counter, const cticp_adaptive_options *adaptive) {
    if (sampling == CTICP_SAMPLING_ADAPTIVE) {
        if (!adaptive) throw std::invalid_argument("adaptive options missing");
        AdaptiveSelect(*adaptive, d_frame_, d_frame_lo(), d_frame_src_, d_counts_ + 1, n_, d_keypoints_, d_kp_lo_, d_kp_src_,
                       d_counts_ + 2);
    } else if (sampling == CTICP_SAMPLING_GRID) {
        GridSelect(d_frame_, d_frame_lo(), d_frame_src_, d_counts_ + 1, n_, sample_voxel_size, 0, 0, 0, 0, 0, 0, 0.f,
                   d_keypoints_, d_kp_lo_, d_kp_src_, d_counts_ + 2);
    } else {
        k_copy_points<<<Blocks(n_), 256, 0, stream_>>>(d_frame_, d_frame_lo(), d_frame_src_, d_counts_ + 1, d_keypoints_,
                                                       d_kp_lo_, d_kp_src_, d_counts_ + 2);
        launches_ += 1;
    }
    if (max_num_keypoints > 0) {
        k_truncate_shuffle<<<Blocks(n_), 256, 0, stream_>>>(d_keypoints_, d_keypoints_lo(), d_kp_src_, d_counts_ + 2,
                                                            max_num_keypoints, seed, counter, d_tmp_points_, d_tmp_lo_,
                                                            d_tmp_src_);
        k_clamp_count<<<1, 1, 0, stream_>>>(d_counts_ + 2, max_num_keypoints);
        std::swap(d_keypoints_, d_tmp_points_);
        std::swap(d_kp_lo_, d_tmp_lo_);
        std::swap(d_kp_src_, d_tmp_src_);
        launches_ += 2;
    }
    CT_CUDA_CHECK(cudaGetLastError());
}

void FramePipeline::QueueCountsReadback() {
    CT_CUDA_CHECK(cudaMemcpyAsync(h_counts_, d_counts_, sizeof(int) * 4, cudaMemcpyDeviceToHost, stream_));
}

void FramePipeline::DistortFrame(const Q4 &qb, const V3 &tb, const Q4 &qe, const V3 &te) {
    EnsureLo();
    k_distort_frame<<<Blocks(n_), 256, 0, stream_>>>(d_frame_, d_frame_lo_, frame_lo_ ? 1 : 0, d_counts_ + 1, qb, tb, qe, te,
                                                     slerp_consts(qb, qe));
    frame_lo_ = distorted_ = true;
    launches_ += 1;
    CT_CUDA_CHECK(cudaGetLastError());
}

void FramePipeline::TransformFrame(const Q4 &qb, const V3 &tb, const Q4 &qe, const V3 &te) {
    k_transform_points<<<Blocks(n_), 256, 0, stream_>>>(d_frame_, d_frame_lo(), d_counts_ + 1, qb, tb, qe, te, slerp_consts(qb, qe), d_frame_world_);
    launches_ += 1;
    CT_CUDA_CHECK(cudaGetLastError());
}

void FramePipeline::EnsureAllWorld() {
    if (!d_all_world_) CT_CUDA_CHECK(cudaMalloc(&d_all_world_, sizeof(double) * 3 * max_points_));
}
void FramePipeline::TransformAll(const Q4 &qb, const V3 &tb, const Q4 &qe, const V3 &te, cudaStream_t stream) {
    EnsureAllWorld();
    k_transform_points<<<Blocks(n_), 256, 0, stream ? stream : stream_>>>(raw_, d_raw_lo(), d_counts_ + 0, qb, tb, qe, te, slerp_consts(qb, qe), d_all_world_);
    launches_ += 1;
    CT_CUDA_CHECK(cudaGetLastError());
}

void FramePipeline::TransformInto(const float4 *pts, const float4 *lo, const int *d_n, const Q4 &qb, const V3 &tb,
                                  const Q4 &qe, const V3 &te, double *d_world, cudaStream_t stream) {
    k_transform_points<<<Blocks(n_), 256, 0, stream ? stream : stream_>>>(pts, lo, d_n, qb, tb, qe, te, slerp_consts(qb, qe), d_world);
    launches_ += 1;
    CT_CUDA_CHECK(cudaGetLastError());
}

}  // namespace cticp
