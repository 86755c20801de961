"""Cost of a checkpoint of the bench scene (bench.make_options / bench.make_scans, configs[1]) after --frames frames:
blob size, median wall time of save_state and load_state (each ends in a device synchronise), where that time goes
(device kernels and copies from a torch.profiler trace of one more call each; the checksum as the time of
state_options, which reads the header and checksums the whole blob on the host), and a plain device<->pageable-host
copy of the same number of bytes for comparison. The card's name and power limit are read in the same run.

  python tools/state_roundtrip.py --out state_roundtrip.json [--frames 24] [--repeats 20]"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from profile_kernels import card_info, kernel_short_name  # noqa: E402


def _median_ms(fn, repeats):
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def _device_split(fn):
    """kernel and copy time (us) of one call, by name, from a torch.profiler trace"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    kernels, copies = {}, {}
    for e in trace.get("traceEvents", []):
        if e.get("cat") == "kernel":
            n = kernel_short_name(e["name"])
            kernels[n] = kernels.get(n, 0.0) + float(e["dur"])
        elif e.get("cat") == "gpu_memcpy":
            copies[e["name"]] = copies.get(e["name"], 0.0) + float(e["dur"])
    if not kernels:
        raise RuntimeError("the trace holds no kernel: is a CUDA device present?")
    return {"kernel_us": sum(kernels.values()), "copy_us": sum(copies.values()), "kernels": kernels, "copies": copies}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--frames", type=int, default=24)
    ap.add_argument("--repeats", type=int, default=20)
    args = ap.parse_args()

    import torch

    import ct_icp_b200
    torch.cuda.init()
    card = card_info()
    eng = ct_icp_b200.engine()
    seq = bench.make_scans(args.frames, bench.WORKLOADS["kitti64_gn"][0])
    od = eng.odometry(bench.make_options(eng))
    for s in seq:
        assert od.RegisterFrame(s["xyz"], s["t"], s["frame_idx"]).success
    blob = od.save_state()
    target = eng.odometry(eng.state_options(blob))
    target.load_state(blob)
    assert target.save_state() == blob

    def save():
        od.save_state()

    def load():
        target.load_state(blob)

    for fn in (save, load):   # warm-up (module loading, CUB's first launches)
        fn()
    save_ms = _median_ms(save, args.repeats)
    load_ms = _median_ms(load, args.repeats)
    checksum_ms = _median_ms(lambda: eng.state_options(blob), args.repeats)
    split = {"save": _device_split(save), "load": _device_split(load)}

    n = len(blob)
    dev = torch.empty(n, dtype=torch.uint8, device="cuda")
    host = torch.empty(n, dtype=torch.uint8)   # pageable, like the caller's buffer

    def d2h():
        host.copy_(dev)
        torch.cuda.synchronize()

    def h2d():
        dev.copy_(host)
        torch.cuda.synchronize()

    d2h(), h2d()
    d2h_ms, h2d_ms = _median_ms(d2h, args.repeats), _median_ms(h2d, args.repeats)

    m = od.GetMapPointer()
    levels = bench.make_options(eng).map_options.num_resolutions
    res = {
        "workload": "configs[1] (bench.make_options / bench.make_scans kitti64_gn), state after %d frames" % args.frames,
        "card": card,
        "blob_bytes": n,
        "map_points_per_level": [m.num_points(l) for l in range(levels)],
        "map_voxels_per_level": [m.num_voxels(l) for l in range(levels)],
        "repeats": args.repeats,
        "save_ms_median_min_max": save_ms,
        "load_ms_median_min_max": load_ms,
        "checksum_and_header_ms_median_min_max": checksum_ms,
        "plain_copy_d2h_pageable_ms_median_min_max": d2h_ms,
        "plain_copy_h2d_pageable_ms_median_min_max": h2d_ms,
        "device_split_one_call": split,
    }
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "device_split_one_call"}, indent=1))
    for k in ("save", "load"):
        print(k, "kernels %.1f us, copies %.1f us" % (split[k]["kernel_us"], split[k]["copy_us"]))


if __name__ == "__main__":
    main()
