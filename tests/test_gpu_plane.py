"""GPU tests (-m gpu) of gpdb_sample_above_plane (include/gpd_b200_plane.h): the device fit against the CPU oracle on the
config-3 cloud, the preprocessed raw config-3 scene and krylon, and the cfg key `sample_above_plane` end to end through
detect_grasps, its --sis and --gpus modes and the detectGraspsInCloud C interface.

Bars: winning hypothesis, its inlier count and its coefficients bit-equal (integer counts, the same float32 operations).
The refined coefficients go through pcl::eigen33, whose three libm calls (atan2f, cosf, sinf) are correctly rounded on
the device and glibc's on the host (the caveat of the normal estimation, tests/test_gpu_preprocess.py): a difference of
at most 1e-6 is allowed and printed. Off-plane indices identical, or differing only at points within 1e-6 of the
threshold."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import load_weights
from gpd_b200 import abi, lib, scenes
import plane_oracle
from oracle import oracle
from test_host_cpp import GraspStruct, _host_lib, _write_detector_cfg, write_pcd

pytestmark = pytest.mark.gpu

HOST = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpd_b200", "host")
CLI = os.path.join(HOST, "detect_grasps")


@pytest.fixture(scope="module")
def cli():
    subprocess.check_call(["make", "-C", HOST, "-s"], env={**os.environ, "CXX": "g++"})
    return CLI


def assert_device_equals_oracle(xyz, got, want, threshold=0.01):
    (ig, info_g), (io, info_o) = got, want
    assert info_g["hypothesis"] == info_o["hypothesis"] >= 0
    assert info_g["hypothesis_inliers"] == info_o["hypothesis_inliers"]
    assert np.array_equal(info_g["hypothesis_coefficients"], info_o["hypothesis_coefficients"])
    assert info_g["refined"] == info_o["refined"]
    dc = float(np.abs(info_g["coefficients"].astype(np.float64) - info_o["coefficients"]).max())
    assert dc <= 1e-6, dc
    diff = np.setxor1d(ig, io)
    if len(diff):
        c = info_o["coefficients"].astype(np.float64)
        dist = np.abs(xyz[diff].astype(np.float64) @ c[:3] + c[3])
        assert np.abs(dist - threshold).max() <= 1e-6, dist
    print(f"N={len(xyz)} h={info_g['hypothesis']} inliers={info_g['inliers']} coefficient diff={dc:.3g} "
          f"differing indices={len(diff)}")
    return dc, len(diff)


def _clouds():
    yield "config3", scenes.synthetic_table_scene(3), False
    yield "raw_config3", scenes.synthetic_raw_scene(3), True
    yield "krylon", scenes.krylon_cloud(), False


def test_device_equals_oracle():
    ctx = lib.Context(lib.default_params(channels=15))
    for name, s, raw in _clouds():
        if raw:
            xyz = ctx.preprocess(s["xyz"], s["cam_source"], s["view_points"], lib.preprocess_params())["xyz"]
            assert len(xyz) > 500000
        else:
            xyz = s["xyz"]
            ctx.set_cloud(xyz, s["normals"], s["cam_source"], s["view_points"])
        for M in (1024, 48):
            pp = lib.plane_params(num_hypotheses=M)
            got = ctx.sample_above_plane(pp)
            want = plane_oracle.sample_above_plane(xyz, abi.default_plane_params(num_hypotheses=M))
            print(name, M, end=": ")
            assert_device_equals_oracle(xyz, got, want)
            assert len(got[0]) > 0 and np.all(np.diff(got[0]) > 0)
    ctx.close()


def test_repeat_calls_are_bit_identical_and_errors_are_reported():
    ctx = lib.Context(lib.default_params(channels=15))
    with pytest.raises(lib.GpdbError) as e:
        ctx.sample_above_plane()
    assert e.value.code == -3
    s = scenes.synthetic_table_scene(3)
    ctx.set_cloud(s["xyz"], s["normals"], s["cam_source"], s["view_points"])
    a, ia = ctx.sample_above_plane()
    for _ in range(3):
        b, ib = ctx.sample_above_plane()
        assert np.array_equal(a, b)
        for k in ia:
            assert np.array_equal(np.asarray(ia[k]), np.asarray(ib[k])), k
    for bad in (dict(distance_threshold=0.0), dict(num_hypotheses=0), dict(num_hypotheses=(1 << 20) + 1)):
        with pytest.raises(lib.GpdbError) as e:
            ctx.sample_above_plane(lib.plane_params(**bad))
        assert e.value.code == -1
    # failure cases: a plane only (every point an inlier), two points (no triple)
    g = np.stack(np.meshgrid(np.arange(30), np.arange(30), indexing="ij"), -1).reshape(-1, 2).astype(np.float32) * np.float32(0.01)
    flat = np.column_stack([g, np.full(len(g), 0.5, np.float32)])
    ctx.set_cloud(flat, np.tile([0.0, 0.0, -1.0], (len(flat), 1)))
    idx, info = ctx.sample_above_plane()
    assert len(idx) == 0 and info["inliers"] == len(flat)
    ctx.set_cloud(flat[:2], np.tile([0.0, 0.0, -1.0], (2, 1)))
    idx, info = ctx.sample_above_plane()
    assert len(idx) == 0 and info["hypothesis"] == -1
    ctx.close()


def lcg_draw(plane, k):
    """Cloud::subsample over plane indices: k draws with replacement by the shim's fixed-seed LCG (all when k >= count)."""
    if k <= 0 or k >= len(plane):
        return np.asarray(plane, np.int32)
    s, out = 42, []
    for _ in range(k):
        s = (s * 1664525 + 1013904223) & 0xFFFFFFFF
        out.append(plane[s % len(plane)])
    return np.array(out, np.int32)


def small_table():
    return scenes.synthetic_table_scene(3, n_points=30000)


def device_plane(s):
    ctx = lib.Context(lib.default_params(channels=15))
    ctx.set_cloud(s["xyz"], s["normals"], s["cam_source"], s["view_points"])
    plane, _ = ctx.sample_above_plane()
    ctx.close()
    return plane


def test_detect_grasps_cli_samples_above_the_plane(cli, tmp_path):
    """detect_grasps with sample_above_plane = 1 on a synthetic table: the shim fits the plane on the device, draws its
    samples from the off-plane indices, and the candidates at exactly those samples (count of the filtered candidates,
    best score) equal the oracle's."""
    s = small_table()
    write_pcd(tmp_path / "t.pcd", s["xyz"], s["normals"], binary=True)
    w, _ = load_weights(15)
    cfg = _write_detector_cfg(tmp_path, w, "num_samples = 400\nmin_inliers = 0\nnum_selected = 20\nsample_above_plane = 1\n")
    out = subprocess.check_output([cli, cfg, str(tmp_path / "t.pcd")]).decode()
    plane = device_plane(s)
    assert f" Plane fit succeeded. {len(plane)} samples above plane." in out
    assert 0 < len(plane) < 0.7 * len(s["xyz"])
    sidx = lcg_draw(plane, 400)
    oc = oracle.OracleCloud(s["xyz"], s["normals"], None, np.zeros((1, 3)))
    ro = oc.detect(abi.default_params(15), oracle.WeightPack(w), sidx)
    n_cand = int([l for l in out.splitlines() if "gripper width" in l][0].split(":")[1].split()[0])
    best = float([l for l in out.splitlines() if l.startswith("RESULT")][0].split("best_score=")[1])
    assert n_cand == ro["n_candidates"] > 0
    assert abs(best - ro["candidates"]["score"].max()) <= 1e-4 * abs(best)
    # without the key the samples come from the whole cloud (the table included): a different candidate set
    cfg0 = _write_detector_cfg(tmp_path, w, "num_samples = 400\nmin_inliers = 0\nnum_selected = 20\n")
    out0 = subprocess.check_output([cli, cfg0, str(tmp_path / "t.pcd")]).decode()
    assert "Plane fit" not in out0
    assert int([l for l in out0.splitlines() if "gripper width" in l][0].split(":")[1].split()[0]) != n_cand


def test_sis_cli_samples_above_the_plane(cli, tmp_path):
    """--sis with sample_above_plane = 1: the initial subsample and the uniform draws come from the off-plane indices, so
    every kept position that is a cloud point is an off-plane point; hands and scores at the kept positions equal the
    oracle's."""
    s = small_table()
    write_pcd(tmp_path / "t.pcd", s["xyz"], s["normals"], binary=True)
    w, _ = load_weights(15)
    cfg = _write_detector_cfg(tmp_path, w, "num_samples = 100\nnum_init_samples = 60\nnum_iterations = 3\n"
                              "num_samples_per_iteration = 60\nprob_rand_samples = 0.5\nstandard_deviation = 0.01\n"
                              "min_score = -1000000\nmin_inliers = 0\nnum_selected = 1000\nsample_above_plane = 1\n")
    out = subprocess.check_output([cli, cfg, str(tmp_path / "t.pcd"), "--sis", "3"]).decode()
    assert "Plane fit succeeded." in out
    pos = np.array([[float(x) for x in l.split()[1:]] for l in out.splitlines() if l.startswith("SIS_SAMPLE")])
    grasps = np.array([[float(x) for x in l.split()[1:]] for l in out.splitlines() if l.startswith("SIS_GRASP")])
    plane = device_plane(s)
    on = np.ones(len(s["xyz"]), bool)
    on[plane] = False
    key = {tuple(p): i for i, p in enumerate(s["xyz"].astype(np.float64))}
    hits = [key[tuple(p)] for p in pos if tuple(p) in key]
    assert len(hits) >= 10 and not on[hits].any()
    oc = oracle.OracleCloud(s["xyz"], s["normals"], None, np.zeros((1, 3)))
    ro = oc.detect(abi.default_params(15), oracle.WeightPack(w), oc.set_samples(pos))
    co = ro["candidates"]
    assert len(co) == len(grasps) > 0
    assert np.allclose(co["position"], grasps[:, 1:4], atol=1e-9, rtol=0)
    assert np.abs(co["score"] - grasps[:, 0]).max() <= 1e-4 * np.abs(co["score"]).max()


def test_python_c_interface_samples_above_the_plane(cli, tmp_path):
    """detectGraspsInCloud with sample_above_plane = 1 on the raw points of a synthetic table: every returned grasp was
    found at an off-plane point, and the scores are the best of the library's at the plane-restricted samples."""
    s = small_table()
    raw = np.ascontiguousarray(s["xyz"], np.float32)
    w, _ = load_weights(15)
    cfg = _write_detector_cfg(tmp_path, w, "num_samples = 300\nmin_inliers = 0\nnum_selected = 15\nsample_above_plane = 1\n")
    L = _host_lib(cli)
    cam = np.ones((len(raw), 1), np.int32)
    vp = np.zeros(3, np.float32)
    out = C.POINTER(GraspStruct)()
    n = L.detectGraspsInCloud(cfg.encode(), raw.ctypes.data, cam.ctypes.data, vp.ctypes.data, len(raw), 1, C.byref(out))
    assert n == 15
    ctx = lib.Context(lib.default_params(channels=15))
    ctx.set_weights(w)
    c = ctx.preprocess(raw, cam, np.zeros((1, 3)), lib.preprocess_params(voxelize=0))
    plane, _ = ctx.sample_above_plane()
    assert len(plane) > 0
    off_pts = {tuple(p) for p in c["xyz"][plane].astype(np.float64)}
    for i in range(n):
        assert tuple(out[i].sample[k] for k in range(3)) in off_pts
    r = ctx.detect(lcg_draw(plane, 300))
    best = np.sort(r["candidates"]["score"])[::-1][:n]
    assert np.allclose([out[i].score for i in range(n)], best, rtol=1e-6)
    assert L.freeMemoryGrasps(out) == 0
    ctx.close()


def test_two_gpus_equal_one_with_the_plane_fit(cli, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s = small_table()
    write_pcd(tmp_path / "t.pcd", s["xyz"], s["normals"], binary=True)
    w, _ = load_weights(15)
    cfg = _write_detector_cfg(tmp_path, w, "num_samples = 500\nmin_inliers = 0\nnum_selected = 25\nsample_above_plane = 1\n")
    one = subprocess.check_output([cli, cfg, str(tmp_path / "t.pcd")]).decode()
    two = subprocess.check_output([cli, cfg, str(tmp_path / "t.pcd"), "--gpus", "2"]).decode()
    pick = lambda o: [l for l in o.splitlines() if l.startswith("RESULT") or "Plane fit" in l]
    assert pick(one) == pick(two) and len(pick(one)) == 2
    c1 = [l for l in one.splitlines() if "gripper width" in l][0].split(":")[1].split()[0]
    c2 = [l for l in two.splitlines() if "gripper width" in l][0].split(":")[1].split()[0]
    assert c1 == c2
