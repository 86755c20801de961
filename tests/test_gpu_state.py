"""Checkpoint / resume on the device (include/cticp.h "checkpoint / resume", DESIGN.md §9).

Contract: a run saved after frame k and loaded into a new handle produces the same bits, for every later frame, as the run
that never stopped — and so does the handle that saved and went on, and a handle rewound to the blob. Each configuration
below makes one part of the saved state non-trivial at the split, and the test asserts that it was."""
import struct

import numpy as np
import pytest

import ct_icp_b200
from ct_icp_b200 import _abi as abi
from test_state_format import host_record, map_blob, map_section, pack_key, seal

pytestmark = pytest.mark.gpu


def _options(b, base=None, solver="GN", **overrides):
    o = b.profile(base) if base else b.default_odometry_options()
    o.ct_icp_options.solver = abi.SOLVER[solver]
    o.ct_icp_options.min_number_neighbors = 10
    o.ct_icp_options.ls_max_num_iters = 5
    o.ct_icp_options.ls_num_threads = 8
    o.map_options = b.legacy_map_options(1.0, 20, 0.1)
    o.debug_print = 0
    o.init_num_frames = 3
    for k, v in overrides.items():
        target = o
        *path, last = k.split("__")
        for p in path:
            target = getattr(target, p)
        setattr(target, last, v)
    return o


def _distance_based(o):
    o.neighborhood_strategy.type = 1   # CTICP_STRATEGY_DISTANCE_BASED
    o.map_options.select_valid_normals_direction = 1
    return o


CONFIGS = {
    "gn_continuous": lambda b: _options(b),
    "ceres_driving": lambda b: _options(b, base="default_driving", solver="CERES"),
    "robust_solver": lambda b: _options(b, solver="ROBUST"),
    "adaptive_max_keypoints": lambda b: _options(b, sampling=abi.SAMPLING["ADAPTIVE"], max_num_keypoints=300),
    "distance_based_normals": lambda b: _distance_based(_options(b, solver="CERES")),
    "robust_ladder": lambda b: _options(b, robust_registration=1, robust_num_attempts=3, robust_threshold_ego_orientation=1e-4,
                                        robust_threshold_relative_orientation=1e-4),
    "skipping_tracker": lambda b: _options(b, insertion_ego_rotation_threshold=1e-4, insertion_threshold_frames_skipped=2),
    "grown_tables": lambda b: _options(b, map_options__capacity_voxels=1024),
}
SPLITS = [1, 4]   # inside init_num_frames (3) and after it


def _frame_bits(sm):
    return bytes(sm.frame)


def _record(od, sm):
    return dict(success=int(sm.success), points_added=int(sm.points_added), N=sm.num_all_corrected_points,
                F=sm.num_corrected_points, K=sm.num_keypoints, residuals=sm.number_of_residuals,
                attempts=sm.number_of_attempts, frame=_frame_bits(sm), map_size=od.MapSize())


def _run(od, seq, frames):
    return [_record(od, od.RegisterFrame(seq[i]["xyz"], seq[i]["t"], seq[i]["frame_idx"])) for i in frames]


def _final(od, levels):
    m = od.GetMapPointer()
    return dict(trajectory=[bytes(f) for f in od.Trajectory()], cloud=od.GetMapPointCloud().tobytes(),
                exports=[tuple(a.tobytes() for a in m.export(l)) for l in range(levels)])


_STRAIGHT = {}


def _straight(eng, seq, name):
    if name not in _STRAIGHT:
        o = CONFIGS[name](eng)
        od = eng.odometry(o)
        recs = _run(od, seq, range(len(seq)))
        _STRAIGHT[name] = (recs, _final(od, o.map_options.num_resolutions))
    return _STRAIGHT[name]


def _assert_exercised(name, eng, od, blob, k, recs_before):
    (registered, last_kp, next_level, _fails, _suspect, skipped, _ins, mm_present, _cd, _co) = host_record(blob)
    assert registered == k + 1 and last_kp > 0 and mm_present == 1
    _, m = map_section(blob)
    has_normals, frame_count = struct.unpack_from("<IxxxxQ", m, 32)
    assert frame_count > 0
    if name == "distance_based_normals":
        assert has_normals == 1
    if name == "robust_ladder" and k >= 4:
        assert next_level >= 1
    if name == "skipping_tracker" and k >= 4:
        assert skipped > 0 or not all(r["points_added"] for r in recs_before[1:])
    if name == "grown_tables":
        assert od.GetMapPointer().num_voxels(0) > 512   # above half of the 1024 initial slots: the table grew
    if name == "adaptive_max_keypoints" and k >= 4:
        assert any(r["K"] == 300 for r in recs_before[1:])   # the shuffle-truncation was active


@pytest.mark.parametrize("k", SPLITS)
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_resume_equals_uninterrupted(eng, seq_small, name, k):
    seq = seq_small
    A, A_final = _straight(eng, seq, name)
    o = CONFIGS[name](eng)
    levels = o.map_options.num_resolutions
    B = eng.odometry(o)
    before = _run(B, seq, range(k + 1))
    assert before == A[:k + 1]
    blob = B.save_state()
    _assert_exercised(name, eng, B, blob, k, before)
    assert B.save_state() == blob                             # saving twice: same bytes
    rest = range(k + 1, len(seq))
    B_after = _run(B, seq, rest)

    co = eng.state_options(blob)
    if name == "grown_tables":
        co.map_options.capacity_voxels = 4096
    C = eng.odometry(co)
    C.load_state(blob)
    assert len(C.all_corrected_points()) == 0 and len(C.keypoints()) == 0   # point vectors are not state
    if name != "grown_tables":
        assert C.save_state() == blob                         # save -> load -> save: same bytes
    C_after = _run(C, seq, rest)

    assert B_after == A[k + 1:]
    assert C_after == A[k + 1:]
    assert _final(B, levels) == A_final
    assert _final(C, levels) == A_final

    B.load_state(blob)                                        # rewind a handle that ran to the end
    assert len(B.Trajectory()) == k + 1
    assert _run(B, seq, rest) == A[k + 1:]
    assert _final(B, levels) == A_final


def _points(rng, n, centre):
    return centre + rng.uniform(-8, 8, size=(n, 3))


def _map_equal(a, b, levels, rng):
    for l in range(levels):
        assert a.num_points(l) == b.num_points(l) and a.num_voxels(l) == b.num_voxels(l), l
        xa, va = a.export(l)
        xb, vb = b.export(l)
        assert np.array_equal(xa, xb) and np.array_equal(va, vb), l
    q = rng.uniform(-6, 6, size=(500, 3))
    for x, y in zip(a.compute_neighborhoods(q, 12), b.compute_neighborhoods(q, 12)):
        assert np.array_equal(x, y)
    r = rng.uniform(0.3, 2.0, size=len(q))
    for x, y in zip(a.radius_search(q, r, 12, sensor_location=(1.0, -2.0, 0.5)), b.radius_search(q, r, 12, sensor_location=(1.0, -2.0, 0.5))):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("capacity", [1024, 1 << 16])
def test_standalone_map_roundtrip(eng, capacity):
    rng = np.random.default_rng(7)
    mo = eng.default_map_options()   # three resolutions, normals kept (select_valid_normals_direction)
    mo.capacity_voxels = 2048
    src = eng.voxel_map(mo)
    for i in range(3):
        src.insert(_points(rng, 20000, np.array([i * 2.0, 0, 0])), origin=(i * 2.0, 0.5, 1.0))
    src.remove_far((0.0, 0.0, 0.0), 12.0)
    blob = src.save()
    assert src.save() == blob
    mo2 = eng.default_map_options()
    mo2.capacity_voxels = capacity
    dst = eng.voxel_map(mo2)
    dst.insert(_points(rng, 500, np.zeros(3)))   # replaced entirely by the load
    dst.load(blob)
    assert dst.save() == blob
    _map_equal(src, dst, 3, np.random.default_rng(1))
    for m in (src, dst):
        m.remove_far((3.0, 0.0, 0.0), 9.0)
        m.insert(_points(np.random.default_rng(3), 5000, np.array([5.0, 1.0, 0.0])), origin=(5.0, 1.0, 0.0))
    _map_equal(src, dst, 3, np.random.default_rng(2))


def _level(keys, counts, B=20):
    P = int(sum(counts))
    pts = np.zeros((P, 4), dtype=np.float32)
    pts[:, :3] = 0.1
    pts[:, 3] = 1.0
    return dict(resolution=1.0, min_distance=0.1, B=B, keys=keys, counts=counts, points=pts)


def _bad_map_blob(kind):
    k0, k1, k2 = pack_key(-1, 0, 0), pack_key(0, 0, 0), pack_key(0, 2, -3)
    if kind == "duplicate_key":
        lv = _level([k0, k1, k1], [1, 1, 1])
    elif kind == "unsorted_keys":
        lv = _level([k0, k2, k1], [1, 1, 1])
    elif kind == "sentinel_key":
        lv = _level([k0, k1, (1 << 64) - 2], [1, 1, 1])
    elif kind == "count_above_B":
        lv = _level([k0, k1, k2], [1, 21, 1])
    elif kind == "P_differs":
        lv = _level([k0, k1, k2], [1, 2, 1])
        lv["points"] = lv["points"][:-1]
    else:
        raise AssertionError(kind)
    return map_blob([lv], frame_count=1)


BAD_MAPS = ["duplicate_key", "unsorted_keys", "sentinel_key", "count_above_B", "P_differs"]


@pytest.mark.parametrize("kind", BAD_MAPS)
def test_map_rejects_invalid_blobs(eng, kind):
    mo = eng.legacy_map_options(1.0, 20, 0.1)
    mo.select_valid_normals_direction = 0
    m = eng.voxel_map(mo)
    m.insert(_points(np.random.default_rng(0), 3000, np.zeros(3)))
    before = m.save()
    with pytest.raises(ct_icp_b200.CticpError) as e:
        m.load(_bad_map_blob(kind))
    assert e.value.code == abi.ERR_INVALID_ARGUMENT, str(e.value)
    assert m.save() == before


def test_map_rejects_other_layouts(eng):
    mo = eng.legacy_map_options(1.0, 20, 0.1)
    src = eng.voxel_map(mo)
    src.insert(_points(np.random.default_rng(0), 3000, np.zeros(3)), origin=(0, 0, 0))
    blob = src.save()
    for change in ("resolution", "max_num_points", "min_distance", "normals"):
        o = eng.legacy_map_options(1.0, 20, 0.1)
        if change == "resolution":
            o.resolutions[0].resolution = 0.5
        elif change == "max_num_points":
            o.resolutions[0].max_num_points = 30
        elif change == "min_distance":
            o.resolutions[0].min_distance_between_points = 0.05
        else:
            o.select_valid_normals_direction = 0
        m = eng.voxel_map(o)
        with pytest.raises(ct_icp_b200.CticpError) as e:
            m.load(blob)
        assert e.value.code == abi.ERR_INVALID_ARGUMENT, change
        assert m.num_points(0) == 0


def test_rejected_loads_leave_the_run_untouched(eng, seq_small):
    name, k = "gn_continuous", 4
    A, A_final = _straight(eng, seq_small, name)
    o = CONFIGS[name](eng)
    B = eng.odometry(o)
    _run(B, seq_small, range(k + 1))
    blob = B.save_state()
    # options that differ
    other = CONFIGS[name](eng)
    other.init_num_frames = 4
    D = eng.odometry(other)
    _run(D, seq_small, range(2))
    with pytest.raises(ct_icp_b200.CticpError) as e:
        B.load_state(D.save_state())
    assert e.value.code == abi.ERR_INVALID_ARGUMENT and "init_num_frames" in str(e.value)
    # a map blob with a valid checksum but an invalid content, inside an otherwise valid odometry blob
    off, m = map_section(blob)
    for kind in BAD_MAPS:
        bad = bytearray(blob[:off] + _bad_map_blob(kind))
        struct.pack_into("<Q", bad, 16, len(bad))
        with pytest.raises(ct_icp_b200.CticpError) as e:
            B.load_state(seal(bad))
        assert e.value.code == abi.ERR_INVALID_ARGUMENT, kind
    # damaged bytes
    flipped = bytearray(blob)
    flipped[off + 100] ^= 1
    with pytest.raises(ct_icp_b200.CticpError) as e:
        B.load_state(bytes(flipped))
    assert e.value.code == abi.ERR_INVALID_ARGUMENT
    assert B.save_state() == blob
    assert _run(B, seq_small, range(k + 1, len(seq_small))) == A[k + 1:]
    assert _final(B, o.map_options.num_resolutions) == A_final


def test_state_facade_roundtrip():
    import subprocess
    from test_state_format import build_state_facade
    r = subprocess.run([build_state_facade()], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "STATE FACADE OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
