"""CPU tests of the support-plane fit of `sample_above_plane` (include/gpd_b200_plane.h; Cloud::sampleAbovePlane,
cloud.cpp:407-435): the oracle against a separately written numpy restatement of the specification, against the
ground truth of the synthetic table scene, across seeds and on the failure cases; the host shim's subsample semantics
and cfg handling; the layout of the two new C-ABI structs."""
import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from gpd_b200 import abi, scenes
import plane_oracle
from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "gpd_b200", "host")
MASK64 = (1 << 64) - 1
f32 = np.float32


# ---- numpy restatement of include/gpd_b200_plane.h --------------------------------------------------------------------
def splitmix64(z):
    z = (z + 0x9E3779B97F4A7C15) & MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    return z ^ (z >> 31)


def draw(seed, h, j, n):
    r = splitmix64((splitmix64(seed) + 3 * h + j) & MASK64)
    return ((r >> 32) * n) >> 32


def plane_of_triple(p0, p1, p2):
    with np.errstate(all="ignore"):
        u, v = p1 - p0, p2 - p0  # float32 arrays: every operation rounds to float32
        r = u / v
        if r[0] == r[1] and r[2] == r[1]:
            return None
        a = u[1] * v[2] - u[2] * v[1]
        b = u[2] * v[0] - u[0] * v[2]
        c = u[0] * v[1] - u[1] * v[0]
        s = (a * a + b * b) + c * c
        if not s > 0:
            return None
        n = np.sqrt(s)
        a, b, c = a / n, b / n, c / n
        return np.array([a, b, c, -((a * p0[0] + b * p0[1]) + c * p0[2])], f32)


def inliers(coef, xyz, threshold):
    v = ((coef[0] * xyz[:, 0] + coef[1] * xyz[:, 1]) + coef[2] * xyz[:, 2]) + coef[3]
    return np.abs(v).astype(np.float64) < np.float64(threshold)  # float32 distance against the double threshold


def fit_numpy(xyz, threshold=0.01, M=1024, seed=1):
    xyz = np.asarray(xyz, f32)
    N = len(xyz)
    counts = np.full(M, -1, np.int64)
    coefs = {}
    if N >= 3:
        for h in range(M):
            ids = [draw(seed, h, j, N) for j in range(3)]
            if len(set(ids)) < 3:
                continue
            c = plane_of_triple(xyz[ids[0]], xyz[ids[1]], xyz[ids[2]])
            if c is None:
                continue
            coefs[h] = c
            counts[h] = int(inliers(c, xyz, threshold).sum())
    if not coefs:
        return np.zeros(0, np.int32), {"hypothesis": -1, "counts": counts}
    win = int(np.argmax(counts))  # first maximum = lowest h on a tie; invalid ones are -1
    plane = coefs[win].copy()
    refined = 0
    inl = inliers(plane, xyz, threshold)
    n = int(inl.sum())
    if n >= 4:
        p = xyz[inl]  # ascending index order
        x, y, z = p[:, 0], p[:, 1], p[:, 2]
        acc = [np.add.accumulate(t, dtype=f32)[-1] for t in (x * x, x * y, x * z, y * y, y * z, z * z, x, y, z)]
        acc = [a / f32(n) for a in acc]
        cov = np.array([[acc[0] - acc[6] * acc[6], acc[1] - acc[6] * acc[7], acc[2] - acc[6] * acc[8]],
                        [acc[1] - acc[6] * acc[7], acc[3] - acc[7] * acc[7], acc[4] - acc[7] * acc[8]],
                        [acc[2] - acc[6] * acc[8], acc[4] - acc[7] * acc[8], acc[5] - acc[8] * acc[8]]], f32)
        _, v = oracle.pcl_eigen33(cov)
        v = v.astype(f32)
        plane = np.array([v[0], v[1], v[2], -((v[0] * acc[6] + v[1] * acc[7]) + v[2] * acc[8])], f32)
        refined = 1
    off = np.flatnonzero(~inliers(plane, xyz, threshold)).astype(np.int32)
    info = {"hypothesis": win, "hypothesis_inliers": int(counts[win]), "hypothesis_coefficients": coefs[win],
            "coefficients": plane, "refined": refined, "inliers": N - len(off), "counts": counts}
    if len(off) in (0, N):
        off = off[:0]
    return off, info


def small_table(seed, n_table=1500, n_obj=600):
    rng = np.random.default_rng(seed)
    table = np.column_stack([rng.uniform(-0.3, 0.3, n_table), rng.uniform(-0.2, 0.2, n_table),
                             0.8 + rng.normal(0, 0.002, n_table)])
    obj = np.column_stack([rng.uniform(-0.1, 0.1, n_obj), rng.uniform(-0.1, 0.1, n_obj), rng.uniform(0.65, 0.79, n_obj)])
    xyz = np.vstack([table, obj])
    return xyz[rng.permutation(len(xyz))].astype(f32)


@pytest.mark.parametrize("seed,M,threshold", [(0, 64, 0.01), (1, 200, 0.01), (2, 128, 0.004), (3, 96, 0.02)])
def test_oracle_equals_a_numpy_restatement(seed, M, threshold):
    xyz = small_table(seed)
    pp = abi.default_plane_params(num_hypotheses=M, seed=seed * 7919 + 1, distance_threshold=threshold)
    io, info_o = plane_oracle.sample_above_plane(xyz, pp)
    iw, info_w = fit_numpy(xyz, threshold, M, pp.seed)
    assert np.array_equal(info_o["counts"], info_w["counts"])
    assert (info_o["counts"] >= 0).sum() > M // 2
    for k in ("hypothesis", "hypothesis_inliers", "inliers", "refined"):
        assert info_o[k] == info_w[k], k
    assert np.array_equal(info_o["hypothesis_coefficients"], info_w["hypothesis_coefficients"])
    assert np.array_equal(info_o["coefficients"], info_w["coefficients"])
    assert info_o["refined"] == 1 and len(io) > 0
    assert np.array_equal(io, iw)


def _plane_vs_table(info):
    c = info["coefficients"].astype(np.float64)
    angle = np.degrees(np.arccos(min(1.0, abs(c[2]) / np.linalg.norm(c[:3]))))
    return angle, -c[3] / c[2]


def test_ground_truth_on_the_synthetic_table():
    """Config 3 (scenes.synthetic_table_scene(3), 300 000 points): the table is the plane z = 0.9 with sigma = 0.5 mm,
    voxelised onto 3 mm voxel corners (its points lie at z = 0.8976 and 0.9006). Oracle run on the development machine
    (seed 1, 1024 hypotheses): refined plane 0.016 degrees from the table's, offset z = 0.89702; 188 762 inliers; every
    point with |z - 0.9| > 0.0125 (111 238 points) is off-plane and every point with |z - 0.8985| < 0.003 an inlier.
    Bars: angle < 0.1 degree, offset within [0.894, 0.9], both classifications without exception."""
    s = scenes.synthetic_table_scene(3)
    idx, info = plane_oracle.sample_above_plane(s["xyz"])
    angle, z0 = _plane_vs_table(info)
    assert angle < 0.1 and 0.894 <= z0 <= 0.9, (angle, z0)
    z = s["xyz"][:, 2].astype(np.float64)
    off = np.zeros(len(z), bool)
    off[idx] = True
    far, band = np.abs(z - 0.9) > 0.0125, np.abs(z - 0.8985) < 0.003
    assert far.sum() > 100000 and band.sum() > 150000
    assert off[far].all() and not off[band].any()
    assert np.all(np.diff(idx) > 0) and info["inliers"] == len(z) - len(idx) and info["refined"] == 1


def test_two_seeds_agree_within_the_bars():
    s = scenes.synthetic_table_scene(3)
    z = s["xyz"][:, 2].astype(np.float64)
    sets = []
    for seed in (1, 987654321):
        idx, info = plane_oracle.sample_above_plane(s["xyz"], abi.default_plane_params(seed=seed))
        angle, z0 = _plane_vs_table(info)
        assert angle < 0.1 and 0.894 <= z0 <= 0.9, (seed, angle, z0)
        off = np.zeros(len(z), bool)
        off[idx] = True
        assert off[np.abs(z - 0.9) > 0.0125].all() and not off[np.abs(z - 0.8985) < 0.003].any()
        sets.append(off)
    assert (sets[0] != sets[1]).mean() < 1e-3


def test_failure_and_edge_cases():
    # fewer than 3 points: no triple
    for n in (0, 1, 2):
        idx, info = plane_oracle.sample_above_plane(np.zeros((n, 3), f32) + np.arange(n)[:, None].astype(f32))
        assert len(idx) == 0 and info["hypothesis"] == -1
    # all points collinear (exact float arithmetic): every triple fails isSampleGood
    t = np.arange(100, dtype=f32)
    idx, info = plane_oracle.sample_above_plane(np.column_stack([t, 2 * t, 3 * t]))
    assert len(idx) == 0 and info["hypothesis"] == -1 and (info["counts"] == -1).all()
    # a cloud that is only a plane: every point is an inlier, the fit fails and the whole cloud stays sampled
    g = np.stack(np.meshgrid(np.arange(30), np.arange(30), indexing="ij"), -1).reshape(-1, 2).astype(f32) * f32(0.01)
    flat = np.column_stack([g, np.full(len(g), 0.5, f32)])
    idx, info = plane_oracle.sample_above_plane(flat)
    assert len(idx) == 0 and info["hypothesis"] >= 0 and info["inliers"] == len(flat) and info["refined"] == 1
    # a winner with fewer than 4 inliers keeps the coefficients of its triple
    pts = np.array([[0, 0, 0], [1, 0, 0.1], [0, 1, 0.3], [0.3, 0.2, 1], [0.9, 0.8, 0.5]], f32)
    idx, info = plane_oracle.sample_above_plane(pts)
    assert info["hypothesis_inliers"] == 3 and info["refined"] == 0
    assert np.array_equal(info["coefficients"], info["hypothesis_coefficients"])
    assert len(idx) == 2 and info["inliers"] == 3
    off_w, info_w = fit_numpy(pts)
    assert np.array_equal(idx, off_w) and info_w["hypothesis"] == info["hypothesis"] and info_w["refined"] == 0
    # bad parameters
    for bad in (dict(distance_threshold=0.0), dict(distance_threshold=float("nan")), dict(num_hypotheses=0),
                dict(num_hypotheses=(1 << 20) + 1)):
        with pytest.raises(RuntimeError):
            plane_oracle.sample_above_plane(pts, abi.default_plane_params(**bad))


def test_float_threshold_decides_like_the_double_comparison():
    """The float32 bound the kernels compare against gives the same answer as PCL's float < double comparison."""
    for t in (0.01, 0.004, 0.02, 0.5, 1e-3):
        tf = np.nextafter(f32(t), f32(np.inf)) if float(f32(t)) < t else f32(t)
        xs = np.nextafter(tf, f32(0)), tf, np.nextafter(tf, f32(1)), f32(t)
        for x in xs:
            assert (x < tf) == (float(x) < t)


def test_plane_struct_layouts_match_the_bindings():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "gpd_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu\n", sizeof(gpdb_plane_params), offsetof(gpdb_plane_params, distance_threshold),
         offsetof(gpdb_plane_params, num_hypotheses), offsetof(gpdb_plane_params, seed));
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(gpdb_plane_info), offsetof(gpdb_plane_info, coefficients),
         offsetof(gpdb_plane_info, hypothesis_coefficients), offsetof(gpdb_plane_info, hypothesis),
         offsetof(gpdb_plane_info, hypothesis_inliers), offsetof(gpdb_plane_info, inliers), offsetof(gpdb_plane_info, refined));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "t"), os.path.join(d, "t.c")])
        nums = list(map(int, subprocess.check_output([os.path.join(d, "t")]).decode().split()))
    P, I = abi.PlaneParams, abi.PlaneInfo
    assert nums[:4] == [C.sizeof(P), P.distance_threshold.offset, P.num_hypotheses.offset, P.seed.offset]
    assert nums[4:] == [C.sizeof(I), I.coefficients.offset, I.hypothesis_coefficients.offset, I.hypothesis.offset,
                        I.hypothesis_inliers.offset, I.inliers.offset, I.refined.offset]


# ---- host shim ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host():
    subprocess.check_call(["make", "-C", HOST, "-s"], env={**os.environ, "CXX": "g++"})
    L = C.CDLL(os.path.join(HOST, "libgpd_host.so"))
    L.gpdSubsample.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    return L


def subsample(L, n_points, plane, num_samples):
    plane = np.ascontiguousarray(plane, np.int32)
    out = np.zeros(max(num_samples, n_points, 1), np.int32)
    n = L.gpdSubsample(n_points, plane.ctypes.data if len(plane) else None, len(plane), num_samples, out.ctypes.data)
    return out[:n].copy()


def lcg(n):
    s, out = 42, []
    for _ in range(n):
        s = (s * 1664525 + 1013904223) & 0xFFFFFFFF
        out.append(s)
    return out


def test_subsample_draws_from_the_plane_indices_with_replacement(host):
    """Cloud::subsampleSampleIndices (cloud.cpp:395-405): num_samples draws with replacement from the plane indices;
    all of them when num_samples >= their count or num_samples = 0 (Cloud::subsample returns early, cloud.cpp:350-353)."""
    plane = np.sort(np.random.default_rng(5).choice(5000, 1000, replace=False)).astype(np.int32)
    got = subsample(host, 5000, plane, 500)
    assert np.array_equal(got, plane[[s % 1000 for s in lcg(500)]])
    assert len(np.unique(got)) < 500 and np.isin(got, plane).all()  # with replacement
    for k in (0, 1000, 1001, 4000):
        assert np.array_equal(subsample(host, 5000, plane, k), plane)


def test_subsample_without_plane_indices_is_unchanged(host):
    """Clouds without plane indices keep the uniform draw without replacement (partial Fisher-Yates, fixed-seed LCG)."""
    n, k = 3000, 700
    perm = np.arange(n)
    for i, s in enumerate(lcg(k)):
        j = i + s % (n - i)
        perm[i], perm[j] = perm[j], perm[i]
    assert np.array_equal(subsample(host, n, [], k), perm[:k])
    assert np.array_equal(subsample(host, n, [], n + 5), np.arange(n))
    assert len(subsample(host, n, [], 0)) == 0


def test_cfg_note_no_longer_names_sample_above_plane(host, tmp_path):
    cli = os.path.join(HOST, "detect_grasps")
    (tmp_path / "a.cfg").write_text("sample_above_plane = 1\n")
    out = subprocess.check_output([cli, "--dump-config", str(tmp_path / "a.cfg")]).decode()
    assert "NOTE" not in out and "sample_above_plane" not in out
    json.loads(out[out.index("{"):out.rindex("}") + 1])
    (tmp_path / "b.cfg").write_text("sample_above_plane = 1\nrefine_normals_k = 5\nremove_outliers = 1\n")
    out = subprocess.check_output([cli, "--dump-config", str(tmp_path / "b.cfg")]).decode()
    note = [l for l in out.splitlines() if l.startswith("NOTE")]
    assert len(note) == 1 and "refine_normals_k" in note[0] and "remove_outliers" in note[0]
    assert "sample_above_plane" not in note[0]
