"""The checkpoint blob format (include/cticp.h "checkpoint / resume", DESIGN.md §9) without a GPU: blobs built by hand
from the documented layout are read by cticp_odometry_state_options, damaged ones are rejected, the new entry points are
exported, and the C++ facade's SaveState / LoadState / StateOptions compile with plain g++.

The builders below are also used by tests/test_gpu_state.py to hand-craft map blobs."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import ct_icp_b200
from ct_icp_b200 import _abi as abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASK64 = (1 << 64) - 1
HOST_RECORD = struct.Struct("<qqiiiiiidd")   # OdoHostRecord up to the motion model's options


def checksum(blob):
    """FNV-1a 64 over bytes [32, total) read as little-endian u64 words, the last one zero-padded."""
    body = bytes(blob[32:])
    body += b"\0" * (-len(body) % 8)
    h = 0xcbf29ce484222325
    for (w,) in struct.iter_unpack("<Q", body):
        h = ((h ^ w) * 0x100000001b3) & MASK64
    return h


def seal(blob):
    blob = bytearray(blob)
    struct.pack_into("<Q", blob, 24, checksum(blob))
    return bytes(blob)


def pack_key(x, y, z):
    b = 1 << 20
    return ((x + b) << 42) | ((y + b) << 21) | (z + b)


def map_blob(levels, frame_count, origins=None):
    """levels: dicts with resolution, min_distance, B, keys (list of u64), counts (list), points ((P, 4) float32 stored
    bits) and, when origins is given (per-voxel normals kept), normals ((V, 4) float64)."""
    has_normals = origins is not None
    out = bytearray(b"CTICPMAP" + struct.pack("<IIQQ", 1, len(levels), 0, 0) + struct.pack("<IIQ", int(has_normals), 0, frame_count))
    if has_normals:
        out += np.asarray(origins, dtype="<f8").reshape(-1).tobytes()
    for lv in levels:
        keys, counts = list(lv["keys"]), list(lv["counts"])
        pts = np.asarray(lv["points"], dtype="<f4").reshape(-1, 4)
        out += struct.pack("<ddiiQQ", lv["resolution"], lv["min_distance"], lv["B"], 0, len(keys), len(pts))
        out += np.asarray(keys, dtype="<u8").tobytes()
        c = np.asarray(counts, dtype="<u4").tobytes()
        out += c + b"\0" * (-len(c) % 8)
        out += pts.tobytes()
        if has_normals:
            out += np.asarray(lv["normals"], dtype="<f8").reshape(-1, 4).tobytes()
    struct.pack_into("<Q", out, 16, len(out))
    return seal(out)


def odometry_blob(options, map_bytes, trajectory=()):
    opts = options.copy()
    out = bytearray(b"CTICPODO" + struct.pack("<IIQQ", 1, C.sizeof(abi.OdometryOptions), 0, 0))
    out += bytes(opts)
    out += HOST_RECORD.pack(len(trajectory), 0, 0, 0, 0, 0, 0, 0, 0.0, 0.0)
    out += bytes(abi.MotionModelOptions()) + bytes(abi.Frame())
    out += struct.pack("<Q", len(trajectory))
    for f in trajectory:
        out += bytes(f)
    out += map_bytes
    struct.pack_into("<Q", out, 16, len(out))
    return seal(out)


def map_section(blob):
    """(offset, bytes) of the map blob inside an odometry blob."""
    T = struct.unpack_from("<Q", blob, 32 + C.sizeof(abi.OdometryOptions) + HOST_RECORD.size + C.sizeof(abi.MotionModelOptions)
                           + C.sizeof(abi.Frame))[0]
    off = 32 + C.sizeof(abi.OdometryOptions) + HOST_RECORD.size + C.sizeof(abi.MotionModelOptions) + C.sizeof(abi.Frame) + 8 \
        + T * C.sizeof(abi.Frame)
    return off, blob[off:]


def host_record(blob):
    return HOST_RECORD.unpack_from(blob, 32 + C.sizeof(abi.OdometryOptions))


def _small_map():
    keys = sorted([pack_key(0, 0, 0), pack_key(-3, 5, 7), pack_key(1, -2, 0)])
    counts = [2, 1, 3]
    pts = np.zeros((6, 4), dtype=np.float32)
    pts[:, :3] = np.linspace(0.01, 0.4, 18).reshape(6, 3)
    pts[:, 3] = [1, 2, -2, 1, 3, -3]
    return map_blob([dict(resolution=0.5, min_distance=0.1, B=20, keys=keys, counts=counts, points=pts)], frame_count=3)


def _options():
    eng = ct_icp_b200.engine()
    o = eng.default_odometry_options()
    o.init_num_frames = 7
    o.shuffle_seed = 0x1234
    o.map_options = eng.legacy_map_options(0.5, 20, 0.1)
    return o


def test_state_options_of_a_hand_built_blob():
    eng = ct_icp_b200.engine()
    o = _options()
    blob = odometry_blob(o, _small_map())
    out = eng.state_options(blob)
    assert out.to_dict() == o.to_dict()
    assert bytes(out) == bytes(o)


def _damaged(kind):
    blob = bytearray(odometry_blob(_options(), _small_map()))
    if kind == "truncated":
        return bytes(blob[:-8])
    if kind == "header_only":
        return bytes(blob[:24])
    if kind == "flipped_payload_byte":
        blob[len(blob) // 2] ^= 0x10
        return bytes(blob)
    if kind == "bad_magic":
        blob[0:8] = b"CTICPMAQ"
        return bytes(blob)
    if kind == "bad_version":
        struct.pack_into("<I", blob, 8, 2)
        return seal(blob)
    if kind == "wrong_sizeof_options":
        struct.pack_into("<I", blob, 12, C.sizeof(abi.OdometryOptions) - 8)
        return seal(blob)
    raise AssertionError(kind)


@pytest.mark.parametrize("kind", ["truncated", "header_only", "flipped_payload_byte", "bad_magic", "bad_version",
                                  "wrong_sizeof_options"])
def test_state_options_rejects_damaged_blobs(kind):
    eng = ct_icp_b200.engine()
    with pytest.raises(ct_icp_b200.CticpError) as e:
        eng.state_options(_damaged(kind))
    assert e.value.code == abi.ERR_INVALID_ARGUMENT, str(e.value)


def test_checksum_covers_every_payload_byte():
    blob = odometry_blob(_options(), _small_map())
    _, m = map_section(blob)
    assert checksum(m) == struct.unpack_from("<Q", m, 24)[0]
    assert struct.unpack_from("<Q", m, 16)[0] == len(m)


def test_checkpoint_symbols_are_exported():
    lib = ct_icp_b200.engine().lib
    for name in ("cticp_odometry_save_state", "cticp_odometry_load_state", "cticp_odometry_state_options", "cticp_map_save",
                 "cticp_map_load"):
        assert hasattr(lib, name), name


STATE_EXE = os.path.join(ROOT, "tests", "cpp", "state_facade_test")


def build_state_facade():
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I",
           os.path.join(ROOT, "ct_icp_b200", "include"), os.path.join(ROOT, "tests", "cpp", "state_facade_test.cpp"),
           "-L", os.path.join(ROOT, "ct_icp_b200"), "-lcticp_b200", "-Wl,-rpath," + os.path.join(ROOT, "ct_icp_b200"),
           "-o", STATE_EXE]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return STATE_EXE


def test_state_facade_compiles_and_fails_loudly_without_gpu():
    import torch
    exe = build_state_facade()
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 42, (r.returncode, r.stdout, r.stderr)
    assert "NO_DEVICE" in r.stdout
