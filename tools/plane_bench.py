"""Device time of gpdb_sample_above_plane (the support-plane fit of `sample_above_plane`, include/gpd_b200_plane.h) on
the config-3 cloud (300 000 points) and on the raw config-3 scene after gpdb_preprocess (~526 000 points), next to the
CPU oracle's time for the same fit. Prints one JSON line.

Timing: a host clock around the call, which ends in a stream synchronise (the off-plane indices are copied back);
median of --calls calls after --warmup calls. hypotheses_per_s = num_hypotheses / that median. The card's name and
power limit are read in the same run. Needs a GPU: without one lib.Context raises."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gpd_b200 import abi, lib, scenes  # noqa: E402
import plane_oracle  # noqa: E402
from oracle import oracle  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?", "?"])[:2] if q.returncode == 0 else ("?", "?")
    return name, power


def measure(ctx, xyz, M, warmup, calls, oracle_runs):
    pp = lib.plane_params(num_hypotheses=M)
    for _ in range(warmup):
        ctx.sample_above_plane(pp)
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        idx, info = ctx.sample_above_plane(pp)
        ts.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.median(ts))
    to = []
    for _ in range(oracle_runs):
        t0 = time.perf_counter()
        io, info_o = plane_oracle.sample_above_plane(xyz, abi.default_plane_params(num_hypotheses=M))
        to.append(time.perf_counter() - t0)
    return {"points": int(len(xyz)), "num_hypotheses": M, "device_ms_median": round(ms, 4),
            "device_ms_min": round(1e3 * min(ts), 4), "device_ms_max": round(1e3 * max(ts), 4),
            "hypotheses_per_s": round(M / (ms * 1e-3), 1), "inlier_fraction": round(info["inliers"] / len(xyz), 6),
            "off_plane": int(len(idx)), "refined": info["refined"],
            "off_plane_equal_to_oracle": bool(np.array_equal(idx, io)),
            "oracle_cpu_s_median": round(float(np.median(to)), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--oracle-runs", type=int, default=3)
    ap.add_argument("--hypotheses", type=int, default=1024)
    args = ap.parse_args()
    name, power = card()
    ctx = lib.Context(lib.default_params(channels=15))
    out = {"metric": "gpdb_sample_above_plane", "gpu": name, "power_limit": power, "oracle_threads": oracle.num_threads(),
           "timing": f"host clock around the synchronous call, median of {args.calls} after {args.warmup} warm-up calls"}
    s = scenes.synthetic_table_scene(3)
    ctx.set_cloud(s["xyz"], s["normals"], s["cam_source"], s["view_points"])
    out["config3"] = measure(ctx, s["xyz"], args.hypotheses, args.warmup, args.calls, args.oracle_runs)
    r = scenes.synthetic_raw_scene(3)
    xyz = ctx.preprocess(r["xyz"], r["cam_source"], r["view_points"], lib.preprocess_params())["xyz"]
    out["raw_config3_preprocessed"] = measure(ctx, xyz, args.hypotheses, args.warmup, args.calls, args.oracle_runs)
    out["raw_config3_preprocess_ms"] = round(float(ctx.preprocess_timings()[5]), 3)
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
