"""Per-kernel device times of steady-state RegisterFrame steps of a bench workload (device-resident input, the path
bench.py's `value` times), from a torch.profiler trace with CUDA activities. Writes one JSON: per kernel the number of
launches per frame and the median / max device time of one launch over the profiled frames, plus the card's name, power
limit and SM clock read in the same run. Times taken under a profiler are for comparing kernels, not bench values.

  python tools/profile_kernels.py --out kernels.json [--frames 40] [--workload kitti64_gn]
(CTICP_ENGINE_LIB selects another build of the engine, as for bench.py.)"""
import argparse
import collections
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def card_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [f.strip() for f in out.split(",")]))


def kernel_short_name(name):
    name = name.split("(")[0]
    return name.split("::")[-1].split("<")[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--frames", type=int, default=40, help="profiled steady-state frames")
    ap.add_argument("--preroll", type=int, default=20, help="start-up frames registered before them (as bench.py)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="kitti64_gn", choices=sorted(bench.WORKLOADS))
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import ct_icp_b200
    torch.cuda.init()
    eng = ct_icp_b200.engine()
    bench._WORKLOAD = args.workload
    first = args.preroll + args.warmup
    seq = bench.make_scans(first + args.frames, bench.WORKLOADS[args.workload][0])
    od = eng.odometry(bench.make_options(eng))
    slots = [od.stage_frame(s["xyz"], s["t"]) for s in seq]
    for i in range(first):
        assert od.RegisterStaged(slots[i], seq[i]["frame_idx"]).success
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(first, first + args.frames):
            assert od.RegisterStaged(slots[i], seq[i]["frame_idx"]).success
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    durs = collections.defaultdict(list)
    for e in trace.get("traceEvents", []):
        if e.get("cat") == "kernel":
            durs[kernel_short_name(e["name"])].append(float(e["dur"]))
    if not durs:
        raise RuntimeError("the trace holds no kernel: is a CUDA device present?")
    kernels = {}
    for name, d in sorted(durs.items(), key=lambda kv: -sum(kv[1])):
        a = np.array(d)
        kernels[name] = {"launches_per_frame": len(a) / args.frames, "median_us": float(np.median(a)),
                         "max_us": float(a.max()), "us_per_frame": float(a.sum() / args.frames)}
    res = {"workload": args.workload, "frames": args.frames, "first_frame": first,
           "engine_lib": os.environ.get("CTICP_ENGINE_LIB", "package build"), "card": card_info(),
           "kernel_us_per_frame": sum(k["us_per_frame"] for k in kernels.values()), "kernels": kernels}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for name, k in kernels.items():
        print("%-28s %5.2f/frame  median %8.2f us  max %8.2f us" % (name, k["launches_per_frame"], k["median_us"], k["max_us"]))


if __name__ == "__main__":
    main()
