"""Option defaults, profiles and shipped configurations pinned on the REFERENCE's own sources (SURVEY §8 row a22): the
fixture tests/golden/reference_defaults.json is extracted from the reference tree by tools/extract_reference_defaults.py
(default member initialisers of the option structs, the enumerators, the assignments of the three profile functions,
config/odometry/*.yaml) — not from the oracle. The engine's cticp_default_* / cticp_profile_* must reproduce it field by
field; fields the boundary does not carry are listed explicitly below."""
import json
import os

import pytest

import ct_icp_b200
from ct_icp_b200 import _abi as abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_defaults.json")
REF = json.load(open(GOLDEN))

ENUM_OF = {   # option field -> the reference enum its value names
    "solver": "CT_ICP_SOLVER", "loss_function": "LEAST_SQUARES", "weighting_scheme": "WEIGHTING_SCHEME",
    "parametrization": "POSE_PARAMETRIZATION", "distance": "ICP_DISTANCE", "motion_compensation": "MOTION_COMPENSATION",
    "initialization": "INITIALIZATION", "sampling": "SAMPLING_OPTION", "model": "MODEL_TYPE",
}
# reference fields with no counterpart at the boundary (outputs for the viewer / logs, pointers replaced by embedded structs,
# the pre-"map_options" topology parameters that Odometry only reads when it is given no map options)
NOT_CARRIED = {
    "CTICPOptions": {"estimate_normal_from_neighborhood", "output_residuals", "output_weights", "output_neighborhood_info",
                     "output_normals", "output_lines", "use_distribution"},
    "OdometryOptions": {"debug_viz", "log_to_file", "log_file_destination", "map_options", "neighborhood_strategy",
                        "size_voxel_map", "max_num_points_in_voxel", "voxel_neighborhood", "max_radius_neighborhood",
                        "min_distance_points"},
}


def ref_value(field, v):
    if isinstance(v, str) and field.split(".")[-1] in ENUM_OF:
        name = v.split("::")[-1]
        return REF["enums"][ENUM_OF[field.split(".")[-1]]][name]
    if isinstance(v, bool):
        return int(v)
    return v


def check_struct(ref_fields, got, not_carried=()):
    missing = {f for f in ref_fields if f not in got}
    assert missing <= set(not_carried), "reference fields the boundary lacks: %s" % sorted(missing - set(not_carried))
    for f, v in ref_fields.items():
        if f in got and f not in not_carried:   # (a pointer member the boundary embeds as a struct is compared on its own)
            assert got[f] == pytest.approx(ref_value(f, v), rel=0, abs=0), (f, got[f], v)


def test_enumerators_are_the_references():
    e = REF["enums"]
    assert abi.SOLVER == e["CT_ICP_SOLVER"] and abi.LOSS == e["LEAST_SQUARES"] and abi.WEIGHTING == e["WEIGHTING_SCHEME"]
    assert abi.PARAMETRIZATION == e["POSE_PARAMETRIZATION"] and abi.DISTANCE == e["ICP_DISTANCE"]
    assert abi.MOTION_COMPENSATION == e["MOTION_COMPENSATION"] and abi.INITIALIZATION == e["INITIALIZATION"]
    assert abi.SAMPLING == e["SAMPLING_OPTION"] and abi.MOTION_MODEL == e["MODEL_TYPE"]


def test_default_options_field_by_field():
    d = ct_icp_b200.default_odometry_options().to_dict()
    check_struct(REF["CTICPOptions"], d["ct_icp_options"], NOT_CARRIED["CTICPOptions"])
    check_struct(REF["OdometryOptions"], d, NOT_CARRIED["OdometryOptions"])
    check_struct(REF["MotionModelOptions"], d["default_motion_model"])
    m = d["map_options"]
    check_struct({k: v for k, v in REF["MapOptions"].items() if k != "resolutions"}, m)
    res = REF["MapOptions"]["resolutions"]
    assert m["num_resolutions"] == len(res)
    for got, (r, dmin, nmax) in zip(m["resolutions"], res):
        assert (got["resolution"], got["min_distance_between_points"], got["max_num_points"]) == (r, dmin, nmax)
    ns = d["neighborhood_strategy"]     # OdometryOptions() installs the nearest-neighbor strategy (odometry.h:152-155)
    check_struct(REF["NeighborStrategyOptions"]["base"], ns)
    check_struct(REF["NeighborStrategyOptions"]["DISTANCE_BASED_STRATEGY"], ns)   # (the distance-based fields keep their defaults)
    assert ns["type"] == abi.STRATEGY["NEAREST_NEIGHBOR_STRATEGY"]
    rp = ct_icp_b200.engine().default_map_options().to_dict()
    assert rp["default_radius"] == REF["MapOptions"]["default_radius"]


@pytest.mark.parametrize("name,fn", [("default_driving", "DefaultDrivingProfile"), ("robust_driving", "RobustDrivingProfile"),
                                     ("robust_outdoor_low_inertia", "DefaultRobustOutdoorLowInertia")])
def test_profiles_are_the_references_assignments(name, fn):
    got = ct_icp_b200.engine().profile(name).to_dict()
    expect = ct_icp_b200.default_odometry_options().to_dict()     # (pinned on the reference by the test above)
    carried = 0
    for path, v in REF["profiles"][fn]:      # in source order: a later assignment overrides an earlier one
        node, keys = expect, path.split(".")
        for k in keys[:-1]:
            node = node.get(k) if isinstance(node, dict) else None
        if node is None or keys[-1] not in node:
            assert keys[-1] in NOT_CARRIED["OdometryOptions"] | NOT_CARRIED["CTICPOptions"], path
            continue
        node[keys[-1]] = ref_value(path, v)
        carried += 1
    assert carried >= 3
    assert got == expect


def test_driving_config_yaml_is_what_the_tests_and_the_bench_register_with():
    """config/odometry/driving_config.yaml (BASELINE.json configs[2]) against the option struct the parity tests build
    (tests/test_gpu_parity.py driving_config)."""
    from test_gpu_parity import driving_config
    got = driving_config(ct_icp_b200.engine()).to_dict()
    y = REF["yaml"]["driving_config"]
    icp = dict(y["ct_icp_options"])
    mm = {k: icp.pop(k) for k in list(icp) if k.startswith("beta_")}       # the YAML nests the motion model's betas here
    check_struct({k: v for k, v in icp.items() if k != "debug_print"}, got["ct_icp_options"], NOT_CARRIED["CTICPOptions"])
    check_struct(mm, got["default_motion_model"])
    top = {k: v for k, v in y.items() if not isinstance(v, dict) and k != "debug_print"}   # (the tests run silent)
    assert not got["debug_print"] and not got["ct_icp_options"]["debug_print"]
    check_struct(top, got, NOT_CARRIED["OdometryOptions"])
    ym = y["map_options"]
    assert got["map_options"]["default_radius"] == ym["default_radius"] and got["map_options"]["num_resolutions"] == len(ym["resolutions"])
    for g, r in zip(got["map_options"]["resolutions"], ym["resolutions"]):
        assert {k: g[k] for k in r} == r
    ys = y["neighborhood_strategy"]
    assert got["neighborhood_strategy"]["type"] == abi.STRATEGY[ys["type"]]
    assert (got["neighborhood_strategy"]["max_num_neighbors"], got["neighborhood_strategy"]["min_num_neighbors"]) == \
        (ys["max_num_neighbors"], ys["min_num_neighbors"])


def test_nclt_config_yaml_against_the_parity_tests_options():
    """config/odometry/nclt_config.yaml (BASELINE.json configs[3]) against tests/test_gpu_parity.py nclt_config — which
    deviates in exactly one documented field: `sampling` (GRID there; the ADAPTIVE sampler of the YAML is exercised by
    test_odometry_nclt_config_adaptive_sampling on the same options)."""
    from test_gpu_parity import nclt_config
    got = nclt_config(ct_icp_b200.engine()).to_dict()
    y = REF["yaml"]["nclt_config"]
    icp = {k: v for k, v in y["ct_icp_options"].items() if k != "debug_print"}
    mm = {k: icp.pop(k) for k in list(icp) if k.startswith("beta_")}
    check_struct(icp, got["ct_icp_options"], NOT_CARRIED["CTICPOptions"])
    check_struct(mm, got["default_motion_model"])
    top = {k: v for k, v in y.items() if not isinstance(v, dict) and k not in ("debug_print", "sampling")}
    check_struct(top, got, NOT_CARRIED["OdometryOptions"])
    assert y["sampling"] == "ADAPTIVE" and got["sampling"] == abi.SAMPLING["GRID"]
    ym = y["map_options"]
    assert got["map_options"]["num_resolutions"] == len(ym["resolutions"])
    for g, r in zip(got["map_options"]["resolutions"], ym["resolutions"]):
        assert {k: g[k] for k in r} == r
    ys = y["neighborhood_strategy"]
    assert got["neighborhood_strategy"]["type"] == abi.STRATEGY[ys["type"]]
    assert (got["neighborhood_strategy"]["max_num_neighbors"], got["neighborhood_strategy"]["min_num_neighbors"]) == \
        (ys["max_num_neighbors"], ys["min_num_neighbors"])
