#!/usr/bin/env python
"""bench.py — the hot path's headline benchmark (BASELINE.json: "grasp candidates/sec end-to-end (15ch)").

One "step" = one pass of the whole path (sample -> local frame -> hand search -> grasp image -> LeNet score)
over the batch of sample indices of a BASELINE config (--config, default 3):

  3 (default) : synthetic 300k-point cluttered cloud (seed 3), num_samples = 100000 PER GPU (weak scaling),
                15-channel images, the reference's 15-channel LeNet weights            (BASELINE configs[2])
  4           : seed-4 cloud, num_samples = 1 000 000 with replacement, FIXED total split over the N GPUs
                (strong scaling), 15-channel                                          (BASELINE configs[3])
  5           : two-camera seed-5 cloud, 12-channel images + the OpenVINO-IR ReLU net, num_samples = 200 000
                fixed total (strong scaling)                                          (BASELINE configs[4])

  value : samples/s with inputs resident in HBM (gpdb_detect_resident; N > 1: gpdb_detect_sharded_resident incl. its
          ncclAllGather), CUDA events on the launching stream, max over ranks
  e2e   : the same through the reference-facing C-ABI call with HOST buffers (gpdb_detect; N > 1: gpdb_detect_sharded):
          H2D of the sample indices, D2H of every result, the all-gather
  N > 1 : one process per GPU (torchrun), ONE context per GPU; the multi-GPU plumbing is INSIDE the C-ABI library:
          gpdb_comm_init (ncclCommInitRank), gpdb_set_cloud_bcast (ncclBroadcast of the cloud from rank 0),
          contiguous sample slices, ONE ncclAllGather of fixed-stride {score, flags} slots. torch.distributed only
          carries the 128-byte NCCL id, the barriers and the max-over-ranks of the timings.
          Outside the timed region rank 0 recomputes a 2048-sample subset on its own GPU and checks the gathered
          flags / scores bit for bit ("parity_check").
  --impl reference : the CPU restatement of the reference path (oracle/, OpenMP on all host cores the process may
          use — NOT OMP_NUM_THREADS, which torchrun sets to 1) on a fixed bounded sample, median of 5.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from gpd_b200 import abi, scenes  # noqa: E402

UNIT = "samples/s (1 sample = 8 hand poses swept, ~1.5 classified)"
CONFIGS = {
    3: {"seed": 3, "two_cameras": False, "channels": 15, "samples": 100000, "scaling": "weak", "relu": 0,
        "metric": "grasp candidates/sec end-to-end (15ch)",
        "workload": "BASELINE config 3 (configs[2], the one north_star's 200k/s target is quoted on): synthetic 300k-pt "
                    "cluttered cloud seed 3, num_samples=100000 per GPU, 15-channel images, reference 15-ch LeNet weights"},
    4: {"seed": 4, "two_cameras": False, "channels": 15, "samples": 1000000, "scaling": "strong", "relu": 0,
        "metric": "grasp candidates/sec end-to-end (15ch)",
        "workload": "BASELINE config 4 (configs[3]): synthetic 300k-pt cluttered cloud seed 4, num_samples=1000000 with "
                    "replacement (default_rng(4).integers), FIXED total sharded over the GPUs, 15-channel images, reference "
                    "15-ch LeNet weights"},
    5: {"seed": 5, "two_cameras": True, "channels": 12, "samples": 200000, "scaling": "strong", "relu": 1,
        "metric": "grasp candidates/sec end-to-end (12ch, two views)",
        "workload": "BASELINE config 5 (configs[4]): two-camera synthetic 300k-pt cloud seed 5, num_samples=200000 with "
                    "replacement, FIXED total sharded over the GPUs, 12-channel images (cfg/image_geometry_12channels.cfg), "
                    "the reference's OpenVINO-IR 12-ch ReLU net"},
}
SAMPLES_PER_GPU = CONFIGS[3]["samples"]


def flops_per_image(ch):
    return {"conv1": 2 * 56 * 56 * 20 * 25 * ch, "conv2": 2 * 24 * 24 * 50 * 500, "ip1": 2 * 7200 * 500 + 2 * 500 * 2}


def load_weights(ch=15):
    z = np.load(os.path.join(ROOT, "gpd_b200", "weights", f"lenet_{ch}ch.npz"))
    names = ["conv1_weights", "conv1_biases", "conv2_weights", "conv2_biases", "ip1_weights", "ip1_biases",
             "ip2_weights", "ip2_biases"]
    return [z[n] for n in names]


def make_workload(n_gpus, samples, config=3):
    """Cloud + the FULL sample-index array of the run. `samples` = per-GPU count for a weak-scaling config (3), the
    fixed total for the strong-scaling configs (4, 5)."""
    cfg = CONFIGS[config]
    cloud = scenes.synthetic_table_scene(cfg["seed"], two_cameras=cfg["two_cameras"])
    ncl = len(cloud["xyz"])
    n_total = samples * n_gpus if cfg["scaling"] == "weak" else samples
    if config == 3 and n_total <= ncl:  # SURVEY 8(d): default_rng(3).choice(N, 100000, replace=False)
        sidx = np.random.default_rng(3).choice(ncl, n_total, replace=False).astype(np.int32)
    else:  # configs 4 / 5, and config 3 beyond the cloud size: with replacement
        sidx = np.random.default_rng(cfg["seed"] if config != 3 else 4).integers(0, ncl, n_total).astype(np.int32)
    return cloud, sidx


def bench_params(config, **over):
    cfg = CONFIGS[config]
    return abi.default_params(cfg["channels"], relu_after_conv=cfg["relu"], **over)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        self.cmd = ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)]
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        busy = sorted(sm)[len(sm) // 2:]
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Cores this process may run on — NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline(cloud, sidx, weights, config=3, sample=4096, repeats=5):
    """Times the CPU restatement of the reference path (oracle/) on a FIXED bounded sample of the same workload: the
    first `sample` sample indices of the step, one warm-up pass + `repeats` timed passes, median reported, with the
    reference's three stage timers (grasp_detector.cpp:313-320). The thread count is passed explicitly."""
    from oracle import oracle

    p = bench_params(config)
    oc = oracle.OracleCloud(cloud["xyz"], cloud["normals"], cloud["cam_source"], cloud["view_points"])
    wp = oracle.WeightPack(weights)
    nt_all = host_threads()
    sub = np.ascontiguousarray(sidx[: min(len(sidx), sample)])
    # SMT siblings can hurt this memory-bound code: probe all logical CPUs and half of them, keep the faster (the CPU
    # arm gets its best configuration)
    cand = [nt_all] + ([nt_all // 2] if nt_all >= 16 else [])
    probe = sub[: min(len(sub), 1024)]
    rates = {}
    for c in cand:
        oc.detect(p, wp, probe[:128], nthreads=c)
        t = time.perf_counter()
        oc.detect(p, wp, probe, nthreads=c)
        rates[c] = len(probe) / (time.perf_counter() - t)
    nt = max(rates, key=rates.get)
    oc.detect(p, wp, sub, nthreads=nt)  # warm-up
    dts, stages, r = [], [], None
    for _ in range(repeats):
        t = time.perf_counter()
        r = oc.detect(p, wp, sub, nthreads=nt)
        dts.append(time.perf_counter() - t)
        stages.append(list(r["stage_seconds"][:3]))
    dt = float(np.median(dts))
    st = np.median(np.array(stages), axis=0)
    vals = sorted(len(sub) / d for d in dts)
    return {"value": len(sub) / dt, "unit": UNIT, "cores": nt, "kind": "port", "host_threads_available": nt_all,
            "runs_samples_per_s": [round(v, 1) for v in vals],
            "stage_seconds": {"candidates": round(float(st[0]), 3), "images": round(float(st[1]), 3), "classify": round(float(st[2]), 3)},
            "sample": f"first {len(sub)} of the step's sample indices ({r['n_candidates']} candidates classified), "
                      f"median of {repeats} passes after one warm-up: {dt:.2f} s per pass on {nt} threads "
                      f"(probe: {', '.join(f'{k} thr {v:.0f}/s' for k, v in rates.items())})"}, r


def bench_preprocess(ctx, hbm_peak, with_cpu):
    """Secondary measurement (SURVEY.md 8(f).1): CandidatesGenerator::preprocessPointCloud on the device —
    NaN / workspace filter, voxelisation at 0.003, normal estimation r = 0.03 — for the RAW cloud of the same scene
    family (seed 3, ~0.9 M points -> ~0.5 M voxels), through gpdb_preprocess with HOST buffers."""
    from gpd_b200 import lib
    raw = scenes.synthetic_raw_scene(3)
    pp = lib.preprocess_params()
    n_out = 0
    for _ in range(2):
        n_out = ctx.preprocess(raw["xyz"], raw["cam_source"], raw["view_points"], pp, read_back=False)
    reps, wall, dev_ms = 3, 0.0, np.zeros(6)
    for _ in range(reps):
        t0 = time.perf_counter()
        ctx.preprocess(raw["xyz"], raw["cam_source"], raw["view_points"], pp, read_back=False)
        wall += time.perf_counter() - t0
        dev_ms += ctx.preprocess_timings()
    wall /= reps
    dev_ms /= reps
    m = len(raw["xyz"])
    out = {"metric": "raw points preprocessed / s (filter + voxelise 0.003 + normals r=0.03), host buffers in, processed cloud resident",
           "value": m / wall, "unit": "raw points/s", "raw_points": m, "processed_points": int(n_out),
           "ms_per_call_wall": round(wall * 1e3, 3),
           "device_ms": {k: round(float(v), 3) for k, v in zip(["upload", "filter", "voxelise", "grid", "normals", "total"], dev_ms)},
           "h2d_bytes_per_call": int(m * (12 + 1))}
    cloud = ctx.get_cloud()
    from oracle import oracle
    oc = oracle.OracleCloud(cloud["xyz"], cloud["normals"], cloud["cam_source"], raw["view_points"])
    probe = np.arange(0, n_out, max(1, n_out // 256))[:256]
    n_nb = float(np.mean([len(oc.radius_search(cloud["xyz"][i], pp.normals_radius)[0]) for i in probe]))
    alg = n_out * (n_nb * 16 + 24)  # float4 gather per neighbour + one float64 normal out
    ach = alg / (dev_ms[4] * 1e-3) / 1e9
    out["k_normals"] = {"ms": round(float(dev_ms[4]), 3), "mean_neighbours": n_nb, "algorithmic_bytes": alg, "GB/s": round(ach, 1),
                        "frac_hbm": round(ach / hbm_peak, 4)}
    if with_cpu:
        t0 = time.perf_counter()
        ro = oracle.preprocess(raw["xyz"], raw["cam_source"], raw["view_points"], pp, nthreads=host_threads())
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": m / dt, "unit": "raw points/s", "cores": host_threads(), "kind": "port",
                               "sample": f"the same {m} raw points, once: {dt:.2f} s (voxelise {ro['seconds'][0]:.2f} s, normals {ro['seconds'][1]:.2f} s)"}
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: the reference itself needs
    PCL / Eigen / OpenCV C++ and cannot be built here) on the box's host cores, same config / metric / unit. Under
    torchrun rank 0 alone runs it. Every step = one cpu_baseline measurement (fixed bounded sample, median of 5)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    samples = args.samples or cfg["samples"]
    cloud, sidx = make_workload(args.gpus, samples, args.config)
    weights = load_weights(cfg["channels"])
    vals, cb = [], None
    for it in range(args.warmup + args.steps):
        cb, _ = cpu_baseline(cloud, sidx, weights, args.config, sample=2048 if it < args.warmup else 4096,
                             repeats=1 if it < args.warmup else 5)
        if it >= args.warmup:
            vals.append(cb["value"])
    v = float(np.median(vals))
    line = {"impl": "reference", "metric": cfg["metric"], "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * len(sidx) / v, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64 geometry / f32 LeNet", "data": "synthetic",
            "config": {"workload": cfg["workload"] + "; CPU restatement of the reference path (oracle/, OpenMP on "
                                   f"{cb['cores']} of {cb['host_threads_available']} host threads); each step times a fixed "
                                   "4096-sample prefix (median of 5 passes) and ms_per_step is extrapolated to the full step",
                       "num_samples": int(len(sidx)), "config": args.config},
            "steps_samples_per_s": [round(x, 1) for x in vals],
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "stage_seconds", "runs_samples_per_s",
                                                "host_threads_available")},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    line["cpu_baseline"]["value"] = v
    print(json.dumps(line))


DUMP_BYTES = 60 * 10**6  # keeps --dump-outputs under 64 MB with the .npy headers


def dump_outputs(d, flags, scores, n_candidates):
    """DIR/<name>.npy of one step's results. When all rows would exceed DUMP_BYTES, a fixed, seeded sample of the rows
    (samples) is written; sample_rows lists them."""
    # pose_scores is NaN where no image was classified (include/gpd_b200.h): those NaNs, at poses pose_flags marks as not
    # classified, are written as 0. Every other score is written as computed, so a value the contract does not allow shows.
    classified = (flags & 3) == 3  # GPDB_POSE_VALID | GPDB_POSE_FILTERED
    scores = np.where(~classified & np.isnan(scores), np.float32(0), scores)
    n, P = flags.shape
    per_row = 2 * 4 * P + 8  # flags and scores as float32, the row number as float64
    rows = np.arange(n)
    if n * per_row > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // per_row, replace=False))
    os.makedirs(d, exist_ok=True)
    for name, a in (("pose_flags", flags[rows].astype(np.float32)), ("pose_scores", scores[rows].astype(np.float32)),
                    ("sample_rows", rows.astype(np.float64)), ("n_candidates", np.array([n_candidates], np.float64))):
        np.save(os.path.join(d, name + ".npy"), a)


def _divert_stdout():
    """Send everything written to file descriptor 1 (Python AND native libraries: NCCL prints its version banner to
    stdout when NCCL_DEBUG >= VERSION) to stderr; the ONE JSON line is printed after _restore_stdout."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _restore_stdout(saved):
    sys.stdout.flush()
    try:
        ctypes.CDLL(None).fflush(None)  # flush C stdio buffers into the diverted descriptor first
    except Exception:
        pass
    os.dup2(saved, 1)
    os.close(saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS), help="BASELINE config (3 weak, 4 / 5 strong scaling)")
    ap.add_argument("--samples", type=int, default=0, help="override: samples per GPU (config 3) / total samples (configs 4, 5)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lenet-impl", type=int, default=0)
    ap.add_argument("--no-preprocess", action="store_true", help="skip the secondary gpdb_preprocess measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (pose_flags, pose_scores [samples, poses] "
                         "as float32; the library's NaN score of a pose with no classified image is written as 0; "
                         "sample_rows, n_candidates), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device path's results; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from gpd_b200 import lib

    cfg = CONFIGS[args.config]
    samples = args.samples or cfg["samples"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    saved_stdout = _divert_stdout()
    final_line = None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's banner / warnings: not on stdout
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    cloud, sidx_all = make_workload(n_gpus, samples, args.config)
    weights = load_weights(cfg["channels"])
    n_all = len(sidx_all)

    params = lib.default_params(channels=cfg["channels"], relu_after_conv=cfg["relu"], device=local, lenet_impl=args.lenet_impl)
    P = params.num_hand_axes * params.num_orientations
    C_img = cfg["channels"]
    ctx = lib.Context(params)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_weights(weights)
    if world > 1:
        # multi-GPU plumbing INSIDE the C-ABI: NCCL communicator of the contexts, cloud broadcast from rank 0
        uid = [lib.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
        if rank == 0:
            ctx.set_cloud_bcast(0, cloud["xyz"], cloud["normals"], cloud["cam_source"], cloud["view_points"])
        else:
            ctx.set_cloud_bcast(0)
        lo, hi, slot_samples = lib.shard_bounds(n_all, rank, world)
    else:
        ctx.set_cloud(cloud["xyz"], cloud["normals"], cloud["cam_source"], cloud["view_points"])
        lo, hi, slot_samples = 0, n_all, n_all
    sidx = np.ascontiguousarray(sidx_all[lo:hi])
    n = len(sidx)

    d_sidx = torch.from_numpy(sidx).to(dev)
    if world > 1:
        slot_b = lib.slot_bytes(slot_samples, P)
        d_gath = torch.zeros(world * slot_b, dtype=torch.uint8, device=dev)
    else:
        d_flags = torch.zeros(n * P, dtype=torch.uint8, device=dev)
        d_scores = torch.zeros(n * P, dtype=torch.float32, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stats = abi.Result()

    def step_resident():
        if world > 1:
            return ctx.detect_sharded_resident(d_sidx.data_ptr(), n, slot_samples, d_gath.data_ptr(), stats)
        return ctx.detect_resident(d_sidx.data_ptr(), n, d_flags.data_ptr(), d_scores.data_ptr(), stats)

    def last_step_outputs():
        """(pose_flags, pose_scores) [n_all, P] as the caller of step_resident receives them; N > 1: decoded from the
        all-gathered slots (include/gpd_b200.h: [scores f32 slot_samples*P][flags u8 slot_samples*P, padded])."""
        if world == 1:
            return d_flags.view(n, P).cpu().numpy(), d_scores.view(n, P).cpu().numpy()
        g = d_gath.cpu().numpy()
        flags, scores = [], []
        for r in range(world):
            lo_r, hi_r, _ = lib.shard_bounds(n_all, r, world)
            s = g[r * slot_b:(r + 1) * slot_b]
            scores.append(s[:4 * slot_samples * P].view(np.float32)[:(hi_r - lo_r) * P])
            flags.append(s[4 * slot_samples * P:][:(hi_r - lo_r) * P])
        return np.concatenate(flags).reshape(n_all, P), np.concatenate(scores).reshape(n_all, P)

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    stage_ms = np.zeros(8)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    ncand = 0
    torch.cuda.synchronize()
    for k in range(args.steps):
        flush.fill_(k)  # evict L2 between timed steps
        ev[k][0].record(stream)
        ncand = step_resident()
        ev[k][1].record(stream)
        launches += int(stats.kernel_launches)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    # the last timed step's results, copied before the serial passes below overwrite the buffers
    outputs = last_step_outputs() if args.dump_outputs and rank == 0 else None
    # per-stage device times from a SERIAL pass (outside the timed region): in the timed steps the hand search of the chunks
    # ahead runs concurrently with images / LeNet of the current chunk, so its stage timers overlap the others
    ctx.set_overlap(0)
    stage_ms[:] = 0
    n_serial = min(args.steps, 3)
    for k in range(n_serial):
        flush.fill_(k)
        step_resident()
        stage_ms += ctx.last_timings()
    torch.cuda.synchronize()
    stage_ms *= args.steps / n_serial  # the code below divides by args.steps
    ctx.set_overlap(1)
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        cnt = torch.tensor([float(ncand)], device=dev, dtype=torch.float64)
        dist.all_reduce(cnt)
        ncand_all = int(cnt.item())
    else:
        ncand_all = ncand
    ms_per_step = total_ms / args.steps
    value = n_all / (ms_per_step * 1e-3)

    # ---- end to end through the public C-ABI call with HOST buffers (gpdb_detect / gpdb_detect_sharded)
    h_all = torch.from_numpy(sidx_all).pin_memory().numpy()
    h_loc = torch.from_numpy(sidx).pin_memory().numpy()
    res = abi.Result()

    def step_e2e():
        if world > 1:
            return ctx.detect_sharded_raw(h_all, res)
        return ctx.detect_raw(h_loc, res)

    for _ in range(2):
        step_e2e()
        lib.free_result(res)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_e2e = 0.0
    d2h = 0
    parity = None
    for k in range(args.steps):
        flush.fill_(k)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        nc = step_e2e()
        t_e2e += time.perf_counter() - t0
        if world > 1:
            d2h = n_all * P * 5 + nc * ctypes.sizeof(abi.Pose)
        else:
            d2h = n * 9 * 8 + n + n * P + n * P * 4 + nc * ctypes.sizeof(abi.Pose)
        if world > 1 and rank == 0 and k == args.steps - 1:
            # parity of the multi-GPU result, outside the timed region: a 2048-sample subset spread over ALL ranks' slices
            # is recomputed on this GPU alone and compared bit for bit with the all-gathered arrays
            g_flags = np.ctypeslib.as_array(res.pose_flags, (n_all, P)).copy()
            g_scores = np.ctypeslib.as_array(res.pose_scores, (n_all, P)).copy()
            pick = np.unique(np.linspace(0, n_all - 1, 2048).astype(np.int64))
            lib.free_result(res)
            one = ctx.detect(sidx_all[pick])
            f_eq = bool(np.array_equal(one["pose_flags"], g_flags[pick]))
            s_eq = bool(np.array_equal(one["pose_scores"].view(np.uint32), g_scores[pick].view(np.uint32)))
            parity = {"samples": int(len(pick)), "ranks_covered": int(len(set(np.searchsorted(
                          [lib.shard_bounds(n_all, r, world)[1] for r in range(world)], pick, side="right")))),
                      "flags_bit_equal": f_eq, "scores_bit_equal": s_eq,
                      "candidates_in_subset": int(np.count_nonzero((g_flags[pick] & 3) == 3)),
                      "how": "rank 0 recomputed the subset single-GPU (gpdb_detect) and compared with the ncclAllGather-ed "
                             "pose_flags / pose_scores of gpdb_detect_sharded"}
            if not (f_eq and s_eq):
                raise SystemExit(f"multi-GPU parity check FAILED: {parity}")
        else:
            lib.free_result(res)
    if world > 1:
        t = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_e2e = float(t.item())
    e2e_value = n_all / (t_e2e / args.steps)
    # the reference-facing call of GraspDetector::detectGrasps proper returns the num_selected best grasps only
    # (selectGrasps, cfg default 100): gpdb_detect_select picks them on the device (secondary number, N = 1)
    e2e_select = None
    if world == 1:
        for _ in range(2):
            ctx.detect_select_raw(h_loc, 100, res)
            lib.free_result(res)
        t_sel = 0.0
        for k in range(args.steps):
            flush.fill_(k)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nsel = ctx.detect_select_raw(h_loc, 100, res)
            t_sel += time.perf_counter() - t0
            lib.free_result(res)
        e2e_select = {"value": n / (t_sel / args.steps), "unit": UNIT, "num_selected": 100, "h2d_bytes_per_step": int(n * 4),
                      "d2h_bytes_per_step": int(nsel * ctypes.sizeof(abi.Pose)),
                      "call": "gpdb_detect_select (detectGrasps + selectGrasps, top-100 picked on the device)"}

    if rank == 0:
        if outputs is not None:
            dump_outputs(args.dump_outputs, *outputs, ncand_all)
        st = stage_ms / args.steps  # per step, this rank
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        # neighbourhood statistics for the algorithmic byte counts (SURVEY.md 8(d)), from the oracle's grid
        from oracle import oracle
        oc = oracle.OracleCloud(cloud["xyz"], cloud["normals"], cloud["cam_source"], cloud["view_points"])
        probe = sidx[:: max(1, n // 256)][:256]
        n_hs = float(np.mean([len(oc.radius_search(cloud["xyz"][i], 0.11)[0]) for i in probe]))
        n_img = float(np.mean([len(oc.radius_search(cloud["xyz"][i], 0.10)[0]) for i in probe]))
        fl = flops_per_image(C_img)
        kernels = {
            "k_hands": {"ms": st[1], "bound": "hbm", "bytes": n * (n_hs * 24 + P * (ctypes.sizeof(abi.Pose) + 1))},
            "k_images": {"ms": st[2], "bound": "hbm", "bytes": ncand * (n_img * 24 + 60 * 60 * C_img + ctypes.sizeof(abi.Pose))},
            "lenet_conv1": {"ms": st[5], "bound": "tensor", "flops": ncand * fl["conv1"]},
            "lenet_conv2": {"ms": st[6], "bound": "tensor", "flops": ncand * fl["conv2"]},
            "lenet_ip": {"ms": st[7], "bound": "tensor", "flops": ncand * fl["ip1"]},
        }
        dom = max(kernels, key=lambda k: kernels[k]["ms"])
        kd = kernels[dom]
        # measured DRAM traffic (ncu --set full capture, profiles/traffic.json: bytes per image / per sample) scaled to
        # the units of one step, like `achieved` (which sums all launches of the kernel in the step)
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom)
            if tj:
                traffic = tj["bytes_per_unit"] * (n if tj["unit"] == "sample" else ncand)
        except Exception:
            pass
        if kd["bound"] == "hbm":
            ach = kd["bytes"] / (kd["ms"] * 1e-3) / 1e9
            roof = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                    "per": "step: all launches of the kernel summed (algorithmic bytes, CUDA-event time, ncu DRAM bytes)",
                    "algorithmic_bytes": kd["bytes"]}
        else:
            ach = kd["flops"] / (kd["ms"] * 1e-3) / 1e12
            roof = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s",
                    "frac": ach / tf_peak, "traffic": traffic, "peak_source": peak_src,
                    "per": "step: all launches of the kernel summed (algorithmic flops, CUDA-event time, ncu DRAM bytes)",
                    "algorithmic_flops": kd["flops"]}
        per_kernel = {}
        for k, v in kernels.items():
            if v["bound"] == "hbm":
                a = v["bytes"] / max(v["ms"], 1e-9) / 1e6
                per_kernel[k] = {"ms_per_step": round(v["ms"], 3), "GB/s": round(a, 1), "frac_hbm": round(a / hbm_peak, 4)}
            else:
                a = v["flops"] / max(v["ms"], 1e-9) / 1e9
                per_kernel[k] = {"ms_per_step": round(v["ms"], 3), "TFLOP/s": round(a, 2), "frac_tensor": round(a / tf_peak, 4)}
        # conv1 issues tcgen05 kind::i8 (3 int8 digit planes stacked along N): its instruction peak, measured on B200 with
        # tools/umma_rate.cu, is 8192 MAC / clock / SM = twice the f16 / bf16 rate (profiles/r02_umma_rate.txt)
        per_kernel["lenet_conv1"]["frac_tensor_int8"] = round(per_kernel["lenet_conv1"]["frac_tensor"] / 2.0, 4)
        per_kernel["lenet_conv1"]["note"] = ("kind::i8: frac_tensor is against the bf16 peak (reference scale), frac_tensor_int8 against "
                                             "2 x that, the measured int8 instruction rate")
        line = {
            "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f64 geometry / f32 LeNet", "data": "synthetic",
            "config": {"workload": cfg["workload"], "config": args.config, "num_samples": n_all, "poses_per_sample": P,
                       "samples_this_rank": n,
                       "parallelism": (f"samples sharded over {world} GPUs inside the C-ABI (gpdb_comm_init / gpdb_set_cloud_bcast / "
                                       "gpdb_detect_sharded): contiguous slices, one ncclAllGather of {score, flags} slots")
                       if world > 1 else "1 GPU",
                       "l2": "512 MB flush write between timed steps; per-step CUDA events summed",
                       "lenet": lib.lib().gpdb_build_info().decode()},
            "rates": {"samples_per_s": value, "poses_evaluated_per_s": value * P,
                      "candidates_classified_per_s": ncand_all / (ms_per_step * 1e-3)},
            "stage_ms_per_step": {"frames": round(st[0], 3), "hand_search": round(st[1], 3), "images": round(st[2], 3),
                                  "lenet": round(st[3], 3), "call_total": round(st[4], 3),
                                  "note": "serial pass (gpdb_set_overlap(0)); the timed steps overlap the hand search of the next "
                                          "chunks with images / LeNet, ms_per_step is their wall time"},
            "kernels": per_kernel,
            "roofline": roof,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int((n_all if world > 1 else n) * 4),
                    "d2h_bytes_per_step": int(d2h),
                    "timing": "wall clock around " + ("gpdb_detect_sharded" if world > 1 else "gpdb_detect") +
                              " (host buffers in, every result out in pinned host memory), max over ranks"},
            "e2e_select": e2e_select,
            "gpu_launches": launches,
            "neighbourhood": {"mean_r0.11": n_hs, "mean_r0.10": n_img, "candidates_per_step": ncand_all},
        }
        if parity is not None:
            line["parity_check"] = parity
        if not args.no_cpu_baseline and world == 1:  # the CPU arm beside our line: at N = 1 only (the other ranks would idle in a barrier)
            cb, _ = cpu_baseline(cloud, sidx_all, weights, args.config)
            line["cpu_baseline"] = cb
        if world == 1 and not args.no_preprocess and args.config == 3:
            line["preprocess"] = bench_preprocess(ctx, hbm_peak, not args.no_cpu_baseline)
        final_line = json.dumps(line)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    _restore_stdout(saved_stdout)
    if final_line is not None:
        print(final_line, flush=True)


if __name__ == "__main__":
    main()
