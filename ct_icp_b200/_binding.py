"""Thin ctypes binding over a shared library that implements the include/cticp.h entry points.

`Binding(lib, prefix)` works for any library exporting `<prefix>odometry_create`, ... — the engine uses
prefix "cticp_"; the test-suite binds the CPU oracle (prefix "orc_") through the same class so both are
driven by identical calls. Nothing in this module computes anything: it marshals numpy arrays and PODs.
"""
import ctypes as C

import numpy as np

from . import _abi as abi


class CticpError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"[{code}] {message}")
        self.code = code


def _as_f64_rows(a, cols):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[1] != cols:
        raise ValueError(f"expected an (n, {cols}) array, got {a.shape}")
    return a


def _save_blob(b, name, h):
    size = b.check(b.fn(name)(h, None, 0))
    buf = C.create_string_buffer(size)
    written = b.check(b.fn(name)(h, buf, size))
    assert written == size, (written, size)
    return buf.raw


class Binding:
    def __init__(self, lib, prefix):
        self.lib = lib
        self.prefix = prefix
        self._declare()

    # ------------------------------------------------------------------------------------------------------
    def fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def has(self, name):
        return hasattr(self.lib, self.prefix + name)

    def _declare(self):
        P = C.POINTER
        vp, i32, i64, u32, u64, dbl, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double, C.c_size_t
        sigs = {
            "last_error": (C.c_char_p, []),
            "default_icp_options": (None, [P(abi.IcpOptions)]),
            "default_map_options": (None, [P(abi.MapOptions)]),
            "default_odometry_options": (None, [P(abi.OdometryOptions)]),
            "legacy_map_options": (None, [P(abi.MapOptions), dbl, C.c_int, dbl]),
            "profile_default_driving": (None, [P(abi.OdometryOptions)]),
            "profile_robust_driving": (None, [P(abi.OdometryOptions)]),
            "profile_robust_outdoor_low_inertia": (None, [P(abi.OdometryOptions)]),
            "odometry_create": (C.c_int, [P(abi.OdometryOptions), C.c_int, P(vp)]),
            "odometry_destroy": (None, [vp]),
            "odometry_register_frame": (C.c_int, [vp, vp, sz, vp, sz, sz, u32, P(abi.Frame), P(abi.Summary)]),
            "odometry_get_points": (i64, [vp, C.c_int, vp, sz]),
            "odometry_trajectory": (i64, [vp, P(abi.Frame), sz]),
            "odometry_map_size": (i64, [vp]),
            "odometry_reset": (C.c_int, [vp]),
            "odometry_map": (vp, [vp]),
            "map_create": (C.c_int, [P(abi.MapOptions), C.c_int, P(vp)]),
            "map_destroy": (None, [vp]),
            "map_insert": (C.c_int, [vp, vp, sz, sz]),
            "map_insert_from": (C.c_int, [vp, vp, sz, sz, vp]),
            "map_radius_search": (C.c_int, [vp, vp, vp, sz, C.c_int, vp, vp, vp]),
            "map_remove_far": (C.c_int, [vp, P(dbl), dbl]),
            "map_num_points": (i64, [vp, C.c_int]),
            "map_num_voxels": (i64, [vp, C.c_int]),
            "map_export": (i64, [vp, C.c_int, vp, vp, sz]),
            "map_compute_neighborhoods": (C.c_int, [vp, vp, sz, C.c_int, vp, vp]),
            "map_clear": (C.c_int, [vp]),
            "icp_register": (C.c_int, [vp, P(abi.IcpOptions), P(abi.StrategyOptions), vp, sz, P(abi.Frame),
                                       P(abi.Frame), P(abi.MotionModelOptions), P(abi.IcpSummary)]),
            "icp_gn_normal_equations": (C.c_int, [vp, P(abi.IcpOptions), vp, sz, P(abi.Frame), P(abi.Frame),
                                                  P(abi.MotionModelOptions), vp, vp, P(i32)]),
            "grid_sample_indices": (i64, [C.c_int, vp, sz, sz, dbl, vp, sz]),
            "permutation": (C.c_int, [u64, u64, u32, vp]),
            "adaptive_sample_indices": (i64, [C.c_int, P(abi.AdaptiveOptions), vp, sz, sz, vp, sz]),
            "default_adaptive_options": (None, [P(abi.AdaptiveOptions)]),
            # engine only
            "abi_version": (u32, []),
            "abi_sizeof": (sz, [C.c_char_p]),
            "odometry_map_points": (i64, [vp, vp, sz]),
            "odometry_last_timing": (C.c_int, [vp, P(abi.DeviceTiming)]),
            "nccl_unique_id": (C.c_int, [vp]),
            "odometry_stage_frame": (i64, [vp, vp, sz, vp, sz, sz]),
            "odometry_register_cloud": (C.c_int, [vp, P(abi.CloudView), u32, P(abi.Frame), P(abi.Summary)]),
            "odometry_stage_cloud": (i64, [vp, P(abi.CloudView)]),
            "odometry_write_points": (i64, [vp, C.c_int, P(abi.CloudSink)]),
            "odometry_register_staged": (C.c_int, [vp, i64, u32, P(abi.Summary)]),
            "odometry_clear_staged": (C.c_int, [vp]),
            "odometry_timer_start": (C.c_int, [vp]),
            "odometry_timer_stop": (C.c_int, [vp, P(dbl)]),
            "odometry_flush_l2": (C.c_int, [vp, sz]),
            "odometry_set_gather_timing": (C.c_int, [vp, C.c_int]),
            "odometry_set_summary_points": (C.c_int, [vp, C.c_int]),
            "odometry_register_frame_ex": (C.c_int, [vp, vp, sz, vp, sz, sz, u32, P(abi.Frame), P(abi.MotionPrior), P(abi.Summary)]),
            "odometry_set_callback": (C.c_int, [vp, abi.EVENT_FN, vp]),
            "odometry_reset_options": (C.c_int, [vp, P(abi.OdometryOptions)]),
            "odometry_enable_sharding": (C.c_int, [vp, vp, C.c_int, C.c_int]),
            "odometry_sharding_mode": (C.c_int, [vp]),
            "odometry_save_state": (i64, [vp, vp, sz]),
            "odometry_load_state": (C.c_int, [vp, C.c_char_p, sz]),
            "odometry_state_options": (C.c_int, [C.c_char_p, sz, P(abi.OdometryOptions)]),
            "map_save": (i64, [vp, vp, sz]),
            "map_load": (C.c_int, [vp, C.c_char_p, sz]),
            # oracle only (KAT taps)
            "odometry_last_counters": (None, [vp, P(u64), P(u64)]),
            "neighborhood_describe": (C.c_int, [vp, sz, vp, P(dbl), P(dbl), P(dbl), vp]),
            "pose_transform": (C.c_int, [P(abi.Frame), P(dbl), dbl, P(dbl)]),
            "se3_inverse": (None, [vp, vp, vp, vp]),
            "se3_mul": (None, [vp, vp, vp, vp, vp, vp]),
            "angular_distance": (dbl, [vp, vp]),
            "se3_interpolate": (None, [vp, vp, vp, vp, dbl, vp, vp]),
            "se3_apply": (None, [vp, vp, vp, vp]),
            "ct_point_to_plane_residual": (dbl, [dbl, vp, vp, vp, dbl, vp, vp, vp, vp, vp]),
            "ct_residual": (dbl, [C.c_int, dbl, vp, vp, vp, vp, dbl, vp, vp, vp, vp, vp]),
            "loss_evaluate": (None, [P(abi.IcpOptions), dbl, vp]),
            "corrector": (None, [dbl, vp, P(dbl), P(dbl)]),
            "quat_plus": (None, [vp, vp, vp]),
            "lm_solve_plane_blocks": (None, [P(abi.IcpOptions), C.c_int, vp, vp, vp, vp, vp, vp, vp]),
            "quat_from_matrix": (None, [vp, vp]),
            "quat_to_matrix": (None, [vp, vp]),
            "symmetric_svd3": (None, [vp, vp, vp]),
            "ldlt_solve12": (None, [vp, vp, vp]),
        }
        for name, (res, args) in sigs.items():
            if self.has(name):
                f = self.fn(name)
                f.restype = res
                f.argtypes = args

    def check(self, code):
        if code < 0:
            msg = self.fn("last_error")()
            raise CticpError(code, msg.decode("utf-8", "replace") if msg else "")
        return code

    # ---- options -------------------------------------------------------------------------------------------
    def default_odometry_options(self):
        o = abi.OdometryOptions()
        self.fn("default_odometry_options")(C.byref(o))
        return o

    def default_icp_options(self):
        o = abi.IcpOptions()
        self.fn("default_icp_options")(C.byref(o))
        return o

    def default_map_options(self):
        o = abi.MapOptions()
        self.fn("default_map_options")(C.byref(o))
        return o

    def legacy_map_options(self, size_voxel_map=1.0, max_num_points_in_voxel=20, min_distance_points=0.1):
        o = abi.MapOptions()
        self.fn("legacy_map_options")(C.byref(o), size_voxel_map, max_num_points_in_voxel, min_distance_points)
        return o

    def profile(self, name):
        o = abi.OdometryOptions()
        self.fn("profile_" + name)(C.byref(o))
        return o

    # ---- factories -----------------------------------------------------------------------------------------
    def odometry(self, options, device=0):
        return Odometry(self, options, device)

    def voxel_map(self, options, device=0):
        return VoxelMap(self, options=options, device=device)

    # ---- sampling ------------------------------------------------------------------------------------------
    def grid_sample_indices(self, xyz, voxel_size, device=0):
        xyz = _as_f64_rows(xyz, 3)
        out = np.empty(len(xyz), dtype=np.uint32)
        n = self.check(self.fn("grid_sample_indices")(device, xyz.ctypes.data, 24, len(xyz), voxel_size,
                                                       out.ctypes.data, len(out)))
        return out[:n].copy()

    def adaptive_sample_indices(self, xyz, options=None, device=0):
        xyz = _as_f64_rows(xyz, 3)
        if options is None:
            options = abi.AdaptiveOptions()
            self.fn("default_adaptive_options")(C.byref(options))
        out = np.empty(len(xyz) + 1, dtype=np.uint32)
        n = self.check(self.fn("adaptive_sample_indices")(device, C.byref(options), xyz.ctypes.data, 24, len(xyz),
                                                           out.ctypes.data, len(out)))
        return out[:n].copy()

    def state_options(self, blob):
        """The effective options stored in an odometry state blob (Odometry.save_state); no device needed."""
        blob = bytes(blob)
        o = abi.OdometryOptions()
        self.check(self.fn("odometry_state_options")(blob, len(blob), C.byref(o)))
        return o

    def permutation(self, seed, counter, n):
        out = np.empty(n, dtype=np.uint32)
        self.check(self.fn("permutation")(seed, counter, n, out.ctypes.data))
        return out


class VoxelMap:
    """ct_icp::MultipleResolutionVoxelMap (include/ct_icp/map.h:99-606) behind the C ABI."""

    def __init__(self, binding, options=None, device=0, borrowed_handle=None, owner=None):
        self.b = binding
        self._owner = owner
        self._borrowed = borrowed_handle is not None
        # the oracle hands out a heap wrapper even for borrowed maps; the engine returns an interior pointer
        self._free_wrapper = self._borrowed and binding.prefix == "orc_"
        if borrowed_handle is not None:
            self.h = C.c_void_p(borrowed_handle)
        else:
            self.h = C.c_void_p()
            binding.check(binding.fn("map_create")(C.byref(options), device, C.byref(self.h)))

    def close(self):
        if self.h and (not self._borrowed or self._free_wrapper):
            self.b.fn("map_destroy")(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def insert(self, xyz, origin=None):          # InsertPointCloud, map.h:153-254 (origin = frame_poses.front().tr)
        xyz = _as_f64_rows(xyz, 3)
        if origin is None:
            self.b.check(self.b.fn("map_insert")(self.h, xyz.ctypes.data, 24, len(xyz)))
        else:
            o = (C.c_double * 3)(*[float(v) for v in origin])
            self.b.check(self.b.fn("map_insert_from")(self.h, xyz.ctypes.data, 24, len(xyz), o))

    def remove_far(self, location, distance):    # RemoveElementsFarFromLocation, map.h:305-322
        loc = (C.c_double * 3)(*location)
        self.b.check(self.b.fn("map_remove_far")(self.h, loc, distance))

    def num_points(self, map_idx=0):
        return self.b.check(self.b.fn("map_num_points")(self.h, map_idx))

    def num_voxels(self, map_idx=0):
        return self.b.check(self.b.fn("map_num_voxels")(self.h, map_idx))

    def export(self, map_idx=0):
        """Returns (xyz (P,3) f64, voxel (P,3) i32), sorted by (voxel, insertion order)."""
        n = self.num_points(map_idx)
        xyz = np.empty((n, 3), dtype=np.float64)
        vox = np.empty((n, 3), dtype=np.int32)
        m = self.b.check(self.b.fn("map_export")(self.h, map_idx, xyz.ctypes.data, vox.ctypes.data, n))
        assert m == n, (m, n)
        return xyz, vox

    def compute_neighborhoods(self, queries, max_num_neighbors=20):
        q = _as_f64_rows(queries, 3)
        pts = np.zeros((len(q), max_num_neighbors, 3), dtype=np.float64)
        cnt = np.zeros(len(q), dtype=np.int32)
        self.b.check(self.b.fn("map_compute_neighborhoods")(self.h, q.ctypes.data, len(q), max_num_neighbors,
                                                            pts.ctypes.data, cnt.ctypes.data))
        return pts, cnt

    def radius_search(self, queries, radiuses, max_num_neighbors=20, sensor_location=None):
        """ComputeNeighborhoods(queries, radiuses, max_num_neighbors, true, sensor_location), map.h:434-447."""
        q = _as_f64_rows(queries, 3)
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(radiuses, dtype=np.float64), (len(q),)))
        pts = np.zeros((len(q), max_num_neighbors, 3), dtype=np.float64)
        cnt = np.zeros(len(q), dtype=np.int32)
        loc = (C.c_double * 3)(*[float(v) for v in sensor_location]) if sensor_location is not None else None
        self.b.check(self.b.fn("map_radius_search")(self.h, q.ctypes.data, r.ctypes.data, len(q), max_num_neighbors, loc,
                                                    pts.ctypes.data, cnt.ctypes.data))
        return pts, cnt

    def clear(self):
        self.b.check(self.b.fn("map_clear")(self.h))

    def save(self):
        """The whole map as a canonical blob (bytes); see include/cticp.h, checkpoint / resume."""
        return _save_blob(self.b, "map_save", self.h)

    def load(self, blob):
        """Replaces the map by a blob of `save` (same resolutions and normals; any capacity)."""
        blob = bytes(blob)
        self.b.check(self.b.fn("map_load")(self.h, blob, len(blob)))

    # CT_ICP_Registration::Register(map, keypoints, frame, motion_model), ct_icp.cpp:1026-1037
    def icp_register(self, icp_options, keypoints, frame, previous_frame=None, motion_options=None,
                     strategy=None):
        """keypoints: structured array of abi.wpoint_dtype() (world rewritten in place); frame: abi.Frame (in/out).
        Returns abi.IcpSummary."""
        assert keypoints.dtype == abi.wpoint_dtype() and keypoints.flags.c_contiguous
        summary = abi.IcpSummary()
        st = strategy if strategy is not None else abi.StrategyOptions(0, 20, 8, 0)
        self.b.check(self.b.fn("icp_register")(
            self.h, C.byref(icp_options), C.byref(st), keypoints.ctypes.data, len(keypoints), C.byref(frame),
            C.byref(previous_frame) if previous_frame is not None else None,
            C.byref(motion_options) if motion_options is not None else None, C.byref(summary)))
        return summary

    def gn_normal_equations(self, icp_options, keypoints, frame, previous_frame=None, motion_options=None):
        assert keypoints.dtype == abi.wpoint_dtype() and keypoints.flags.c_contiguous
        A = np.zeros((12, 12))
        b = np.zeros(12)
        n = C.c_int32(0)
        self.b.check(self.b.fn("icp_gn_normal_equations")(
            self.h, C.byref(icp_options), keypoints.ctypes.data, len(keypoints), C.byref(frame),
            C.byref(previous_frame) if previous_frame is not None else None,
            C.byref(motion_options) if motion_options is not None else None, A.ctypes.data, b.ctypes.data,
            C.byref(n)))
        return A, b, n.value


class Odometry:
    """ct_icp::Odometry (include/ct_icp/odometry.h:159-402) behind the C ABI.

    Method names follow the reference: RegisterFrame, RegisterFrameWithEstimate, Trajectory, MapSize,
    GetMapPointCloud, Reset, GetMapPointer."""

    def __init__(self, binding, options, device=0):
        self.b = binding
        self.options = options.copy()
        self.h = C.c_void_p()
        binding.check(binding.fn("odometry_create")(C.byref(self.options), device, C.byref(self.h)))

    def close(self):
        if self.h:
            self.b.fn("odometry_destroy")(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _register(self, xyz, timestamps, frame_id, initial_estimate):
        xyz = np.asarray(xyz)
        timestamps = np.asarray(timestamps)
        if xyz.dtype != np.float64 or xyz.ndim != 2 or xyz.shape[1] < 3 or xyz.strides[1] != 8:
            xyz = np.ascontiguousarray(xyz[:, :3], dtype=np.float64)
        if timestamps.dtype != np.float64 or timestamps.ndim != 1:
            timestamps = np.ascontiguousarray(timestamps, dtype=np.float64).reshape(-1)
        if len(xyz) != len(timestamps):
            raise ValueError("xyz and timestamps must have the same length")
        summary = abi.Summary()
        self.b.check(self.b.fn("odometry_register_frame")(
            self.h, xyz.ctypes.data, xyz.strides[0], timestamps.ctypes.data, timestamps.strides[0], len(xyz),
            frame_id, C.byref(initial_estimate) if initial_estimate is not None else None, C.byref(summary)))
        return summary

    def RegisterFrame(self, xyz, timestamps, frame_id, motion_model=None):
        """motion_model: an abi.MotionPrior — the AMotionModel* of the reference's overloads (odometry.h:231-248)"""
        if motion_model is not None:
            return self._register_ex(xyz, timestamps, frame_id, None, motion_model)
        return self._register(xyz, timestamps, frame_id, None)

    def _register_ex(self, xyz, timestamps, frame_id, initial_estimate, motion_model):
        xyz = np.ascontiguousarray(np.asarray(xyz)[:, :3], dtype=np.float64)
        timestamps = np.ascontiguousarray(timestamps, dtype=np.float64).reshape(-1)
        summary = abi.Summary()
        self.b.check(self.b.fn("odometry_register_frame_ex")(
            self.h, xyz.ctypes.data, xyz.strides[0], timestamps.ctypes.data, timestamps.strides[0], len(xyz), frame_id,
            C.byref(initial_estimate) if initial_estimate is not None else None,
            C.byref(motion_model) if motion_model is not None else None, C.byref(summary)))
        return summary

    def RegisterCallback(self, fn):
        """fn(event) -> bool, called at BEFORE_ITERATION / ITERATION_COMPLETED / FINISHED_REGISTRATION
        (Odometry::RegisterCallback, odometry.h:260); None removes it."""
        self._callback = abi.EVENT_FN(lambda event, user: 1 if fn(event) else 0) if fn else abi.EVENT_FN()
        self.b.check(self.b.fn("odometry_set_callback")(self.h, self._callback, None))

    def ResetWithOptions(self, options):        # Odometry::Reset(const OdometryOptions&), odometry.h:269
        self.options = options.copy()
        self.b.check(self.b.fn("odometry_reset_options")(self.h, C.byref(self.options)))

    def RegisterFrameWithEstimate(self, xyz, timestamps, initial_estimate, frame_id):
        return self._register(xyz, timestamps, frame_id, initial_estimate)

    # ---- record buffers (sensor_msgs/PointCloud2-like), zero-copy in and out (engine only) -------------------
    @staticmethod
    def _cloud_view(records, xyz_field="x", t_field="t"):
        """records: 1-D numpy structured array with fields x, y, z (contiguous, same float type) and a timestamp."""
        assert records.ndim == 1 and records.flags.c_contiguous and records.dtype.fields is not None
        f = records.dtype.fields
        xdt, xoff = f[xyz_field][0], f[xyz_field][1]
        assert f["y"] == (xdt, xoff + xdt.itemsize) and f["z"] == (xdt, xoff + 2 * xdt.itemsize), "x, y, z must be contiguous"
        tdt, toff = f[t_field][0], f[t_field][1]
        return abi.CloudView(records.ctypes.data, len(records), records.dtype.itemsize, xoff, abi.DTYPE[xdt.name], toff,
                             abi.DTYPE[tdt.name], 0)

    def RegisterCloud(self, records, frame_id, initial_estimate=None, t_field="t"):
        """RegisterFrame(const slam::PointCloud&, frame_id) on an interleaved record buffer, read in place."""
        view = self._cloud_view(records, t_field=t_field)
        summary = abi.Summary()
        self.b.check(self.b.fn("odometry_register_cloud")(
            self.h, C.byref(view), frame_id, C.byref(initial_estimate) if initial_estimate is not None else None,
            C.byref(summary)))
        return summary

    def stage_cloud(self, records, t_field="t"):
        view = self._cloud_view(records, t_field=t_field)
        return self.b.check(self.b.fn("odometry_stage_cloud")(self.h, C.byref(view)))

    def write_points(self, which, records, world=True, t_field="t"):
        """Fills `records` (structured array with x, y, z [+ timestamp field]) with one of the summary's point vectors;
        returns the number of points the vector holds."""
        f = records.dtype.fields
        xdt, xoff = f["x"][0], f["x"][1]
        has_t = t_field in f
        sink = abi.CloudSink(records.ctypes.data, len(records), records.dtype.itemsize, xoff, abi.DTYPE[xdt.name],
                             f[t_field][1] if has_t else 0, abi.DTYPE[f[t_field][0].name] if has_t else 0,
                             1 if world else 0)
        return self.b.check(self.b.fn("odometry_write_points")(self.h, which, C.byref(sink)))

    # ---- device-resident input / measurement helpers (engine only) ---------------------------------------
    def stage_frame(self, xyz, timestamps):
        xyz = np.ascontiguousarray(np.asarray(xyz)[:, :3], dtype=np.float64)
        timestamps = np.ascontiguousarray(timestamps, dtype=np.float64).reshape(-1)
        return self.b.check(self.b.fn("odometry_stage_frame")(self.h, xyz.ctypes.data, xyz.strides[0],
                                                              timestamps.ctypes.data, 8, len(xyz)))

    def RegisterStaged(self, slot, frame_id):
        summary = abi.Summary()
        self.b.check(self.b.fn("odometry_register_staged")(self.h, slot, frame_id, C.byref(summary)))
        return summary

    def clear_staged(self):
        self.b.check(self.b.fn("odometry_clear_staged")(self.h))

    def timer_start(self):
        self.b.check(self.b.fn("odometry_timer_start")(self.h))

    def timer_stop(self):
        ms = C.c_double(0.0)
        self.b.check(self.b.fn("odometry_timer_stop")(self.h, C.byref(ms)))
        return ms.value

    def flush_l2(self, nbytes=256 << 20):
        self.b.check(self.b.fn("odometry_flush_l2")(self.h, nbytes))

    def set_gather_timing(self, on):
        self.b.check(self.b.fn("odometry_set_gather_timing")(self.h, 1 if on else 0))

    def set_summary_points(self, mask):
        """bit POINTS_* set: every RegisterFrame produces that vector of the RegistrationSummary eagerly."""
        self.b.check(self.b.fn("odometry_set_summary_points")(self.h, int(mask)))

    def points_into(self, which, buf):
        """one of the summary's point vectors into a caller-owned record array (abi.wpoint_dtype()); returns the count"""
        return self.b.check(self.b.fn("odometry_get_points")(self.h, which, buf.ctypes.data, len(buf)))

    def points(self, which):
        cap = 1 << 16
        while True:
            buf = np.zeros(cap, dtype=abi.wpoint_dtype())
            n = self.b.check(self.b.fn("odometry_get_points")(self.h, which, buf.ctypes.data, cap))
            if n <= cap:
                return buf[:n].copy()
            cap = int(n)

    def corrected_points(self):
        return self.points(abi.POINTS_CORRECTED)

    def all_corrected_points(self):
        return self.points(abi.POINTS_ALL_CORRECTED)

    def keypoints(self):
        return self.points(abi.POINTS_KEYPOINTS)

    def Trajectory(self):
        n = self.b.check(self.b.fn("odometry_trajectory")(self.h, None, 0))
        arr = (abi.Frame * max(n, 1))()
        self.b.check(self.b.fn("odometry_trajectory")(self.h, arr, n))
        return [arr[i].copy() for i in range(n)]

    def MapSize(self):
        return self.b.check(self.b.fn("odometry_map_size")(self.h))

    def GetMapPointer(self):
        return VoxelMap(self.b, borrowed_handle=self.b.fn("odometry_map")(self.h), owner=self)

    def GetMapPointCloud(self):
        xyz, _ = self.GetMapPointer().export(0)
        return xyz

    def Reset(self):
        self.b.check(self.b.fn("odometry_reset")(self.h))

    def save_state(self):
        """Everything that influences the frames to come, as a canonical blob (bytes)."""
        return _save_blob(self.b, "odometry_save_state", self.h)

    def load_state(self, blob):
        """Replaces this handle's state by a blob of save_state (options must match, see Binding.state_options)."""
        blob = bytes(blob)
        self.b.check(self.b.fn("odometry_load_state")(self.h, blob, len(blob)))

    def last_timing(self):
        t = abi.DeviceTiming()
        self.b.check(self.b.fn("odometry_last_timing")(self.h, C.byref(t)))
        return t

    def enable_sharding(self, unique_id_bytes, rank, world):
        buf = (C.c_char * 128).from_buffer_copy(unique_id_bytes)
        self.b.check(self.b.fn("odometry_enable_sharding")(self.h, buf, rank, world))

    def sharding_mode(self):
        """0 = single GPU, 1 = NCCL all-reduce per exchange, 2 = in-kernel exchange over NVLink peer mailboxes."""
        return self.b.fn("odometry_sharding_mode")(self.h)
