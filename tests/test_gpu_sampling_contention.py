"""Contended voxels in the grid selection and the map insert, compared exactly with the CPU oracle.

The selection's claim aggregates the bids of a warp's points that share a voxel before it touches the hash grid, and the
map insert skips voxels that are already full and stages its candidates per warp: these cases put many points into one
voxel, end scans off a warp boundary, fill voxels exactly to their capacity and overflow the commit's staging room.
RegisterStaged reads a staged scan in place; it must register exactly what RegisterFrame registers from host arrays."""
import numpy as np
import pytest

from ct_icp_b200 import _abi as abi
from test_gpu_parity import _sequence_options, small_map_options

pytestmark = pytest.mark.gpu


def _same_selection(orc, eng, xyz, voxel):
    a = orc.grid_sample_indices(xyz, voxel)
    b = eng.grid_sample_indices(xyz, voxel)
    assert len(a) == len(b) and np.array_equal(a, b)
    return b


def test_every_point_in_one_voxel(orc, eng):
    rng = np.random.default_rng(3)
    xyz = rng.uniform(0.05, 0.45, size=(40000, 3))
    assert len(_same_selection(orc, eng, xyz, 0.5)) == 1


def test_hot_voxel_among_singletons(orc, eng):
    rng = np.random.default_rng(5)
    hot = rng.uniform(10.05, 10.45, size=(3000, 3))                     # > 1024 points in one voxel
    singles = np.column_stack([np.arange(5000) + 0.25, np.full(5000, -20.25), np.full(5000, 0.25)])   # one per voxel
    xyz = np.concatenate([singles[:2500], hot, singles[2500:]])        # the hot run contiguous: whole warps agree
    sel = _same_selection(orc, eng, xyz, 0.5)
    assert len(sel) == 5001
    # the same points shuffled: the hot voxel's points spread over many warps
    _same_selection(orc, eng, xyz[rng.permutation(len(xyz))], 0.5)


@pytest.mark.parametrize("n", [1, 5, 31, 33, 1000, 4133])
def test_warp_tail(orc, eng, n):
    rng = np.random.default_rng(n)
    xyz = rng.uniform(-2.0, 2.0, size=(n, 3))
    _same_selection(orc, eng, xyz, 0.5)
    _same_selection(orc, eng, xyz, 1.5)


def _same_map(mo, me):
    assert mo.num_points() == me.num_points()
    assert mo.num_voxels() == me.num_voxels()
    xo, vo = mo.export()
    xe, ve = me.export()
    assert np.array_equal(vo, ve)
    assert np.abs(xo - xe).max() < 2e-7


def test_map_insert_into_full_voxels(orc, eng):
    """Voxels fill up to exactly B, then more points arrive for them and for fresh voxels."""
    B = 5
    mo = orc.voxel_map(small_map_options(orc, res=1.0, max_pts=B, min_dist=0.05))
    me = eng.voxel_map(small_map_options(eng, res=1.0, max_pts=B, min_dist=0.05))
    rng = np.random.default_rng(9)
    centres = rng.integers(0, 40, size=(300, 3)).astype(np.float64)   # (>= 0: int() truncation merges no voxels)
    # B well-separated points per voxel: every one is accepted
    offs = np.array([[0.1, 0.1, 0.1], [0.3, 0.1, 0.1], [0.1, 0.3, 0.1], [0.1, 0.1, 0.3], [0.3, 0.3, 0.3]])
    first = (centres[:, None, :] + offs[None, :, :]).reshape(-1, 3)
    mo.insert(first)
    me.insert(first)
    _same_map(mo, me)
    assert me.num_points() == B * len(np.unique(centres, axis=0))
    # full voxels receive more (acceptable) points, together with points for new voxels
    late = (centres[:, None, :] + rng.uniform(0.5, 0.95, size=(len(centres), 4, 3))).reshape(-1, 3)
    fresh = rng.uniform(30.0, 40.0, size=(2000, 3))
    for batch in (late, np.concatenate([fresh, late])):
        mo.insert(batch)
        me.insert(batch)
        _same_map(mo, me)


def test_map_insert_more_candidates_than_staging(orc, eng):
    """One voxel with more than 512 candidates in a single insert (the commit's slow path), next to ordinary voxels."""
    mo = orc.voxel_map(small_map_options(orc, res=1.0, max_pts=20, min_dist=0.1))
    me = eng.voxel_map(small_map_options(eng, res=1.0, max_pts=20, min_dist=0.1))
    rng = np.random.default_rng(13)
    crowd = rng.uniform(2.02, 2.98, size=(1500, 3))
    others = rng.uniform(-10.0, 10.0, size=(3000, 3))
    pts = np.concatenate([others[:1000], crowd, others[1000:]]).astype(np.float32).astype(np.float64)
    mo.insert(pts)
    me.insert(pts)
    _same_map(mo, me)


def _frame_values(sm):
    f = sm.frame
    return (list(f.begin_pose.tr) + list(f.begin_pose.quat) + list(f.end_pose.tr) + list(f.end_pose.quat) +
            [sm.success, sm.num_corrected_points, sm.num_keypoints, sm.number_of_residuals, sm.points_added])


def test_register_staged_equals_register_frame(eng, seq_small):
    od_host = eng.odometry(_sequence_options(eng, init_num_frames=3))
    od_dev = eng.odometry(_sequence_options(eng, init_num_frames=3))
    slots = [od_dev.stage_frame(s["xyz"], s["t"]) for s in seq_small]
    for s, slot in zip(seq_small, slots):
        a = od_host.RegisterFrame(s["xyz"], s["t"], s["frame_idx"])
        b = od_dev.RegisterStaged(slot, s["frame_idx"])
        assert _frame_values(a) == _frame_values(b)
        assert od_host.MapSize() == od_dev.MapSize()
    expect = od_host.points(abi.POINTS_ALL_CORRECTED)
    # the last frame's points stay readable after the staged scans are freed
    od_dev.clear_staged()
    got = od_dev.points(abi.POINTS_ALL_CORRECTED)
    for k in expect.dtype.names:
        assert np.array_equal(expect[k], got[k]), k
