"""C++ host shims (gpd_b200/host: the reference's class names over the C-ABI) and the detect_grasps command line.
CPU: cfg and PCD parsing (the reference's caller-side formats, SURVEY 8(f)-2). GPU: the whole CLI against the ctypes path."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from gpd_b200 import scenes
from oracle.reference_data import config_parser_answers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "gpd_b200", "host")
CLI = os.path.join(HOST, "detect_grasps")


@pytest.fixture(scope="module")
def cli():
    subprocess.check_call(["make", "-C", HOST, "-s"], env={**os.environ, "CXX": "g++"})
    return CLI


def write_pcd(path, xyz, normals=None, binary=False):
    n = len(xyz)
    fields = "x y z" + (" normal_x normal_y normal_z" if normals is not None else "")
    k = 6 if normals is not None else 3
    hdr = (f"# .PCD v.7 - Point Cloud Data file format\nVERSION .7\nFIELDS {fields}\nSIZE {' '.join(['4'] * k)}\n"
           f"TYPE {' '.join(['F'] * k)}\nCOUNT {' '.join(['1'] * k)}\nWIDTH {n}\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS {n}\n"
           f"DATA {'binary' if binary else 'ascii'}\n")
    rows = np.hstack([xyz, normals]).astype(np.float32) if normals is not None else np.asarray(xyz, np.float32)
    with open(path, "wb") as f:
        f.write(hdr.encode())
        if binary:
            f.write(rows.tobytes())
        else:
            for r in rows:
                f.write((" ".join(repr(float(v)) for v in r) + "\n").encode())


def test_cfg_and_pcd_parsing(cli, tmp_path):
    (tmp_path / "hand.cfg").write_text("# hand geometry\nfinger_width = 0.012   # comment\nhand_outer_diameter=0.13\nhand_depth = 0.07\n"
                                       "hand_height\t=\t0.025\ninit_bite = 0.015\n")
    (tmp_path / "main.cfg").write_text(
        f"hand_geometry_filename = {tmp_path}/hand.cfg\nimage_geometry_filename = 0\n"
        "volume_width = 0.11\nimage_num_channels = 12\n# defaults for the rest of the image geometry\n"
        "weights_file = /some/where/params/\nnum_samples = 77\nnum_samples = 99\nnum_orientations = 6\nhand_axes = 0 2\n"
        "deepen_hand = 0\nworkspace_grasps = -0.5 0.5 -0.4 0.4 0.1 1.1\nmax_aperture = 0.07\n"
        "filter_approach_direction = 1\ndirection = 0 0 1\nthresh_rad = 1.5\nmin_inliers = 0\nnum_selected = 7\n"
        "voxel_size = 0.004\nworkspace = -0.9 0.9 -0.8 0.8 -0.7 0.7\nnormals_radius = 0.025\nthis line has no separator\n")
    xyz = np.array([[0.1, 0.2, 0.3], [np.nan, 0, 0], [1.5, -2.5, 3.25]], np.float32)
    nrm = np.array([[0, 0, 1], [0, 1, 0], [1, 0, 0]], np.float32)
    for binary in (False, True):
        write_pcd(tmp_path / "c.pcd", xyz, nrm, binary=binary)
        out = subprocess.check_output([cli, "--dump-config", str(tmp_path / "main.cfg"), str(tmp_path / "c.pcd")]).decode()
        d = json.loads(out[out.index("{"):out.rindex("}") + 1])
        assert (d["finger_width"], d["hand_outer_diameter"], d["hand_depth"], d["hand_height"], d["init_bite"]) == (0.012, 0.13, 0.07, 0.025, 0.015)
        assert (d["volume_width"], d["volume_depth"], d["volume_height"], d["image_size"], d["image_num_channels"]) == (0.11, 0.06, 0.02, 60, 12)
        assert d["num_samples"] == 77  # first occurrence wins (config_file.cpp:44-50)
        assert (d["num_orientations"], d["num_hand_axes"], d["hand_axes0"], d["deepen_hand"]) == (6, 2, 0, 0)
        assert d["workspace_grasps"] == [-0.5, 0.5, -0.4, 0.4, 0.1, 1.1] and d["max_aperture"] == 0.07 and d["min_aperture"] == 0.0
        assert d["filter_approach_direction"] == 1 and d["direction"] == [0, 0, 1] and d["thresh_rad"] == 1.5
        assert d["weights_file"] == "/some/where/params/" and d["num_selected"] == 7 and d["min_inliers"] == 0
        assert d["nn_radius"] == 0.01 and d["num_finger_placements"] == 10 and d["friction_coeff"] == 20 and d["min_viable"] == 6
        assert (d["voxelize"], d["voxel_size"], d["normals_radius"]) == (1, 0.004, 0.025)
        assert d["workspace"] == [-0.9, 0.9, -0.8, 0.8, -0.7, 0.7]
        assert d["cloud_points"] == 2 and d["cloud_has_normals"] == 1  # the NaN point is removed
        assert np.allclose(d["first_point"], [0.1, 0.2, 0.3], atol=1e-7)


@pytest.mark.gpu
def test_detect_grasps_cli_matches_library(cli, tmp_path):
    from conftest import load_weights
    from gpd_b200 import lib
    k = scenes.krylon_cloud()
    write_pcd(tmp_path / "krylon.pcd", k["xyz"], k["normals"], binary=True)
    w, _ = load_weights(15)
    os.makedirs(tmp_path / "params")
    names = ["conv1_weights", "conv1_biases", "conv2_weights", "conv2_biases", "ip1_weights", "ip1_biases", "ip2_weights", "ip2_biases"]
    for n, a in zip(names, w):
        a.astype(np.float32).tofile(tmp_path / "params" / (n + ".bin"))
    (tmp_path / "main.cfg").write_text(f"hand_geometry_filename = 0\nimage_geometry_filename = 0\nweights_file = {tmp_path}/params/\n"
                                       "num_samples = 5000\nmin_inliers = 0\nnum_selected = 10\nimage_num_channels = 15\nvoxelize = 0\n")
    out = subprocess.check_output([cli, str(tmp_path / "main.cfg"), str(tmp_path / "krylon.pcd")]).decode()
    res = [l for l in out.splitlines() if l.startswith("RESULT")][0]
    n_grasps = int(res.split("n_grasps=")[1].split()[0])
    best = float(res.split("best_score=")[1])
    # num_samples >= N: every point is a sample (cloud.cpp:364-370)
    p = lib.default_params(channels=15)
    ctx = lib.Context(p)
    ctx.set_weights(w)
    ctx.set_cloud(k["xyz"], k["normals"], k["cam_source"], k["view_points"])
    r = ctx.detect(np.arange(len(k["xyz"]), dtype=np.int32))
    assert n_grasps == 10
    assert abs(best - r["candidates"]["score"].max()) <= 1e-3 * abs(best)
    assert f"gripper width: {r['n_candidates']}" in out
    ctx.close()


@pytest.mark.gpu
def test_detect_grasps_cli_preprocesses_a_raw_cloud(cli, tmp_path, golden_dir):
    """Raw PCD without normals: the CLI filters, voxelises and estimates normals on the device
    (GraspDetector::preprocessPointCloud -> gpdb_preprocess) and then runs the path; same result as the ctypes
    calls on the same raw points."""
    from conftest import load_weights
    from gpd_b200 import lib
    raw = np.load(os.path.join(golden_dir, "krylon_preprocess.npz"))["raw"]
    write_pcd(tmp_path / "raw.pcd", raw, None, binary=True)
    w, _ = load_weights(15)
    os.makedirs(tmp_path / "params")
    names = ["conv1_weights", "conv1_biases", "conv2_weights", "conv2_biases", "ip1_weights", "ip1_biases", "ip2_weights", "ip2_biases"]
    for n, a in zip(names, w):
        a.astype(np.float32).tofile(tmp_path / "params" / (n + ".bin"))
    (tmp_path / "main.cfg").write_text(f"hand_geometry_filename = 0\nimage_geometry_filename = 0\nweights_file = {tmp_path}/params/\n"
                                       "num_samples = 5000\nmin_inliers = 0\nnum_selected = 10\nimage_num_channels = 15\n"
                                       "centered_at_origin = 1\n")
    out = subprocess.check_output([cli, str(tmp_path / "main.cfg"), str(tmp_path / "raw.pcd")]).decode()
    assert "Voxelized cloud: 2373" in out
    res = [l for l in out.splitlines() if l.startswith("RESULT")][0]
    best = float(res.split("best_score=")[1])
    ctx = lib.Context(lib.default_params(channels=15))
    ctx.set_weights(w)
    c = ctx.preprocess(raw, None, np.zeros((1, 3)), lib.preprocess_params())
    ctx.set_cloud(c["xyz"], -c["normals"], c["cam_source"], c["view_points"])  # centered_at_origin (detect_grasps.cpp:75-80)
    r = ctx.detect(np.arange(len(c["xyz"]), dtype=np.int32))
    assert int(res.split("n_grasps=")[1].split()[0]) == 10
    assert abs(best - r["candidates"]["score"].max()) <= 1e-3 * abs(best)
    ctx.close()


class GraspStruct(__import__("ctypes").Structure):
    """struct Grasp of src/detect_grasps_python.cpp:49-56."""
    import ctypes as _C
    _fields_ = [("pos", _C.POINTER(_C.c_double)), ("orient", _C.POINTER(_C.c_double)), ("sample", _C.POINTER(_C.c_double)),
                ("score", _C.c_double), ("label", _C.c_bool), ("image", _C.POINTER(_C.c_int))]


def _host_lib(cli):
    import ctypes as C
    L = C.CDLL(os.path.join(HOST, "libgpd_host.so"))
    L.detectGraspsInCloud.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.POINTER(GraspStruct))]
    L.detectGraspsInCloudNormals.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                             C.POINTER(C.POINTER(GraspStruct))]
    L.freeMemoryGrasps.argtypes = [C.POINTER(GraspStruct)]
    L.gpdQuaternionFromMatrix.argtypes = [C.c_void_p, C.c_void_p]
    return L


def test_python_c_interface_symbols_and_quaternion(cli):
    """The reference's extern "C" interface for Python callers (detect_grasps_python.cpp:431-475,598-601) is exported
    by libgpd_host.so; the quaternion is Eigen::Quaterniond(Matrix3d) (x, y, z, w; w >= 0 branch when trace > 0)."""
    from scipy.spatial.transform import Rotation
    L = _host_lib(cli)
    rng = np.random.default_rng(0)
    for R in Rotation.random(200, random_state=1).as_matrix():
        m = np.asfortranarray(R)
        q = np.zeros(4)
        L.gpdQuaternionFromMatrix(m.ctypes.data, q.ctypes.data)
        assert abs(np.linalg.norm(q) - 1) < 1e-12
        assert np.allclose(Rotation.from_quat(q).as_matrix(), R, atol=1e-12)
        if np.trace(R) > 0:
            assert q[3] > 0
        else:
            assert q[int(np.argmax(np.diag(R)))] > 0
    assert L.detectGraspsInCloud(None, None, None, None, 0, 0, None) == -1


def test_python_c_interface_file_entry_points_reject_bad_input(cli, tmp_path):
    """detectGraspsInFile / generateGraspCandidatesInFile / detectAndEvalGrasps / CopyAndFree (detect_grasps_python.cpp:468-549,
    603-607) are exported; missing arguments and a missing cloud file give 0 grasps before any device is touched (the reference
    returns 0 when the cloud is empty, :474-476)."""
    import ctypes as C
    L = _host_lib(cli)
    out = C.POINTER(GraspStruct)()
    vp = np.zeros(3, np.float32)
    for f in (L.detectGraspsInFile, L.generateGraspCandidatesInFile):
        f.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_int, C.POINTER(C.POINTER(GraspStruct))]
        assert f(None, None, None, None, 0, None) == 0
        assert f(b"none.cfg", str(tmp_path / "missing.pcd").encode(), b"", vp.ctypes.data, 1, C.byref(out)) == 0
        assert not out
    L.detectAndEvalGrasps.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                      C.POINTER(C.POINTER(GraspStruct))]
    assert L.detectAndEvalGrasps(None, None, None, None, 0, 0, None, None, 0, None) == 0
    L.CopyAndFree.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    assert L.CopyAndFree(None, None, 0) == -1


@pytest.mark.gpu
def test_python_c_interface_detects_like_the_library(cli, tmp_path, golden_dir):
    import ctypes as C
    from conftest import load_weights
    from gpd_b200 import lib
    L = _host_lib(cli)
    raw = np.ascontiguousarray(np.load(os.path.join(golden_dir, "krylon_preprocess.npz"))["raw"], np.float32)
    w, _ = load_weights(15)
    os.makedirs(tmp_path / "params")
    names = ["conv1_weights", "conv1_biases", "conv2_weights", "conv2_biases", "ip1_weights", "ip1_biases", "ip2_weights", "ip2_biases"]
    for n, a in zip(names, w):
        a.astype(np.float32).tofile(tmp_path / "params" / (n + ".bin"))
    (tmp_path / "main.cfg").write_text(f"hand_geometry_filename = 0\nimage_geometry_filename = 0\nweights_file = {tmp_path}/params/\n"
                                       "num_samples = 5000\nmin_inliers = 0\nnum_selected = 25\nimage_num_channels = 15\n")
    cam = np.ones((len(raw), 1), np.int32)
    vp = np.zeros(3, np.float32)
    out = C.POINTER(GraspStruct)()
    n = L.detectGraspsInCloud(str(tmp_path / "main.cfg").encode(), raw.ctypes.data, cam.ctypes.data, vp.ctypes.data, len(raw), 1,
                              C.byref(out))
    assert n == 25
    ctx = lib.Context(lib.default_params(channels=15))
    ctx.set_weights(w)
    c = ctx.preprocess(raw, cam, np.zeros((1, 3)), lib.preprocess_params())
    r = ctx.detect(np.arange(len(c["xyz"]), dtype=np.int32))
    cand = r["candidates"]
    order = np.argsort(-cand["score"], kind="stable")[:25]
    scores = np.array([out[i].score for i in range(n)])
    assert np.allclose(scores, cand["score"][order], rtol=1e-6)
    for i in (0, 7, 24):
        j = order[i]
        if i and scores[i] == scores[i - 1]:
            continue  # ties may be ordered differently by partial_sort
        assert np.allclose([out[i].pos[k] for k in range(3)], cand["position"][j])
        assert np.allclose([out[i].sample[k] for k in range(3)], cand["sample"][j])
        q = np.array([out[i].orient[k] for k in range(4)])
        from scipy.spatial.transform import Rotation
        assert np.allclose(Rotation.from_quat(q).as_matrix(), cand["frame"][j].reshape(3, 3).T, atol=1e-9)
        assert bool(out[i].label) == bool(cand["full_antipodal"][j]) and out[i].image[0] == -1
    assert L.freeMemoryGrasps(out) == 0
    ctx.close()


@pytest.mark.gpu
def test_python_c_interface_candidates_and_eval_entry_points(cli, tmp_path, golden_dir):
    """detectAndEvalGrasps (candidates + images + labels against a ground-truth cloud) and the library calls it composes:
    the hands equal gpdb_hand_search's candidates on the preprocessed cloud, the images gpdb_images', the labels
    gpdb_reevaluate's against the ground-truth cloud."""
    import ctypes as C
    from conftest import load_weights
    from gpd_b200 import lib
    L = _host_lib(cli)
    raw = np.ascontiguousarray(np.load(os.path.join(golden_dir, "krylon_preprocess.npz"))["raw"], np.float32)
    w, _ = load_weights(15)
    os.makedirs(tmp_path / "params")
    names = ["conv1_weights", "conv1_biases", "conv2_weights", "conv2_biases", "ip1_weights", "ip1_biases", "ip2_weights", "ip2_biases"]
    for n, a in zip(names, w):
        a.astype(np.float32).tofile(tmp_path / "params" / (n + ".bin"))
    (tmp_path / "main.cfg").write_text(f"hand_geometry_filename = 0\nimage_geometry_filename = 0\nweights_file = {tmp_path}/params/\n"
                                       "num_samples = 5000\nmin_inliers = 0\nnum_selected = 25\nimage_num_channels = 15\n")
    cam = np.ones((len(raw), 1), np.int32)
    vp = np.zeros(3, np.float32)
    ctx = lib.Context(lib.default_params(channels=15))
    ctx.set_weights(w)
    c = ctx.preprocess(raw, cam, np.zeros((1, 3)), lib.preprocess_params())
    sidx = np.arange(len(c["xyz"]), dtype=np.int32)
    cand = ctx.hand_search(sidx)["candidates"]
    imgs = ctx.images(cand)
    gt_xyz = np.ascontiguousarray(c["xyz"][::2], np.float32)  # a thinned copy of the processed cloud as "ground truth"
    gt_nrm = np.ascontiguousarray(c["normals"][::2], np.float32)
    L.detectAndEvalGrasps.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                      C.POINTER(C.POINTER(GraspStruct))]
    out = C.POINTER(GraspStruct)()
    n = L.detectAndEvalGrasps(str(tmp_path / "main.cfg").encode(), raw.ctypes.data, cam.ctypes.data, vp.ctypes.data, len(raw), 1,
                              gt_xyz.ctypes.data, gt_nrm.ctypes.data, len(gt_xyz), C.byref(out))
    assert n == len(cand) > 0
    ctx.set_cloud(gt_xyz, gt_nrm.astype(np.float64), None, np.zeros((1, 3)))
    labels, _ = ctx.reevaluate(cand)
    isz = imgs[0].size
    for i in (0, n // 2, n - 1):
        assert np.allclose([out[i].pos[k] for k in range(3)], cand["position"][i])
        assert bool(out[i].label) == bool(labels[i])
        assert np.array_equal(np.ctypeslib.as_array(out[i].image, (isz,)), imgs[i].ravel().astype(np.int32))
    assert L.freeMemoryGrasps(out) == 0
    ctx.close()


def test_clustering_matches_a_python_restatement(cli):
    """Clustering::findClusters (clustering.cpp:5-105) in the host shim against a line-by-line numpy restatement."""
    import ctypes as C
    from gpd_b200 import abi
    L = C.CDLL(os.path.join(HOST, "libgpd_host.so"))
    L.gpdFindClusters.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    rng = np.random.default_rng(4)
    n = 120
    hands = np.zeros(n, dtype=abi.POSE_DTYPE)
    centers = rng.uniform(-0.1, 0.1, (6, 3))
    axes = rng.standard_normal((6, 3))
    axes /= np.linalg.norm(axes, axis=1, keepdims=True)
    for i in range(n):
        c = i % 6
        a = axes[c] + rng.normal(0, 0.02, 3)
        a /= np.linalg.norm(a)
        hands["frame"][i][6:9] = a                                   # Hand::getAxis = third column
        hands["position"][i] = centers[c] + a * rng.uniform(-0.03, 0.03) + rng.normal(0, 0.001, 3)
        hands["score"][i] = rng.normal(100, 30)
        hands["full_antipodal"][i] = i % 2

    def restate(min_inliers, remove):
        out, used = [], np.zeros(n, bool)
        for i in range(n):
            ai, pi = hands["frame"][i][6:9], hands["position"][i]
            k, pos, mean, sd = 0, np.zeros(3), 0.0, 0.0
            for j in range(n):
                if i == j or (remove and used[j]):
                    continue
                aj, pj = hands["frame"][j][6:9], hands["position"][j]
                d = pi - pj
                proj = (np.eye(3) - np.outer(ai, ai)) @ d
                if abs(ai @ aj) > np.cos(np.deg2rad(12.0)) and np.linalg.norm(d) <= 0.05 and np.linalg.norm(proj) <= 0.005:
                    k += 1
                    pos += pj
                    old, sj = mean, float(hands["score"][j])
                    mean += (sj - mean) / k
                    sd += (sj - mean) * (sj - old)
                    if remove:
                        used[j] = True
            if k >= min_inliers:
                sd /= k
                sd = np.sqrt(sd) if sd != 0 else sd
                out.append((i, pi + (pos / k - pi), mean - 2.576 * sd / np.sqrt(k)))
        return out

    for min_inliers, remove in ((1, 0), (3, 0), (2, 1), (0, 0)):
        got = np.zeros(n, dtype=abi.POSE_DTYPE)
        m = L.gpdFindClusters(hands.ctypes.data, n, min_inliers, remove, got.ctypes.data)
        exp = restate(min_inliers, remove)
        assert m == len(exp)
        for g, (i, pos, lb) in zip(got[:m], exp):
            assert np.allclose(g["position"], pos, atol=1e-12) and abs(g["score"] - np.float32(lb)) <= 1e-4 * max(1, abs(lb))
            assert np.array_equal(g["frame"], hands["frame"][i]) and g["full_antipodal"] == hands["full_antipodal"][i]


def test_shipped_cfg_files_parse_like_the_reference(cli, golden_dir):
    """The reference's own cfg files (copies in tests/golden/cfg; relative geometry / model paths resolved from the working
    directory, as upstream does) through the shim's parser: eigen_params.cfg, vino_params_12channels.cfg,
    all_axes_vino_12channels.cfg."""
    def dump(name):
        out = subprocess.check_output([cli, "--dump-config", name], cwd=os.path.join(golden_dir, "cfg")).decode()
        return json.loads(out[out.index("{"):out.rindex("}") + 1])
    d = dump("eigen_params.cfg")
    assert (d["image_num_channels"], d["num_samples"], d["num_selected"], d["min_inliers"]) == (15, 30, 5, 0)
    assert d["weights_file"] == "../models/lenet/15channels/params/" and d["voxelize"] == 1 and d["voxel_size"] == 0.003
    assert (d["finger_width"], d["hand_outer_diameter"], d["hand_depth"], d["hand_height"], d["init_bite"]) == (0.01, 0.12, 0.06, 0.02, 0.01)
    d = dump("vino_params_12channels.cfg")
    assert (d["image_num_channels"], d["num_hand_axes"], d["hand_axes0"], d["min_inliers"], d["num_selected"]) == (12, 1, 2, 1, 50)
    assert d["weights_file"].endswith("two_views_12_channels_curv_axis.bin")
    d = dump("all_axes_vino_12channels.cfg")
    assert (d["image_num_channels"], d["num_hand_axes"], d["hand_axes0"]) == (12, 3, 0)


def _lzf_compress(data):
    """Minimal LZF encoder for the test (greedy, 3-byte hash table): literals + back references, format of liblzf."""
    out, lit, i, n, table = bytearray(), bytearray(), 0, len(data), {}

    def flush():
        nonlocal lit
        while lit:
            chunk, lit = lit[:32], lit[32:]
            out.append(len(chunk) - 1)
            out.extend(chunk)
    while i < n:
        key = bytes(data[i:i + 3])
        ref = table.get(key) if len(key) == 3 else None
        table[key] = i
        if ref is not None and 0 < i - ref <= 8192:
            ln = 3
            while i + ln < n and ln < 264 and data[ref + ln] == data[i + ln]:
                ln += 1
            flush()
            dist, l2 = i - ref - 1, ln - 2
            if l2 < 7:
                out.append((l2 << 5) | (dist >> 8))
            else:
                out.append((7 << 5) | (dist >> 8))
                out.append(l2 - 7)
            out.append(dist & 255)
            i += ln
        else:
            lit.append(data[i])
            i += 1
    flush()
    return bytes(out)


def test_ply_and_compressed_pcd_readers(cli, tmp_path):
    """Cloud::loadPointCloudFromFile reads .pcd and .ply (cloud.cpp:643-660): PLY ascii / binary_little_endian and PCD
    binary_compressed (LZF, field-major payload) give the same cloud as the plain binary PCD."""
    rng = np.random.default_rng(2)
    xyz = np.round(rng.uniform(-1, 1, (300, 3)), 2).astype(np.float32)  # repeated byte patterns: back references occur
    xyz[7] = [np.nan, 0, 0]
    nrm = rng.standard_normal((300, 3)).astype(np.float32)
    (tmp_path / "main.cfg").write_text("weights_file = /x/\n")

    def dump(path):
        out = subprocess.check_output([cli, "--dump-config", str(tmp_path / "main.cfg"), str(path)]).decode()
        d = json.loads(out[out.index("{"):out.rindex("}") + 1])
        return d["cloud_points"], d["cloud_has_normals"], d.get("first_point")
    write_pcd(tmp_path / "plain.pcd", xyz, nrm, binary=True)
    ref = dump(tmp_path / "plain.pcd")
    assert ref[0] == 299 and ref[1] == 1
    # PCD binary_compressed
    soa = np.concatenate([np.hstack([xyz, nrm])[:, k] for k in range(6)]).astype(np.float32).tobytes()
    comp = _lzf_compress(soa)
    assert len(comp) < len(soa)
    hdr = ("# .PCD v.7\nVERSION .7\nFIELDS x y z normal_x normal_y normal_z\nSIZE 4 4 4 4 4 4\nTYPE F F F F F F\nCOUNT 1 1 1 1 1 1\n"
           "WIDTH 300\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS 300\nDATA binary_compressed\n")
    open(tmp_path / "lzf.pcd", "wb").write(hdr.encode() + struct.pack("<II", len(comp), len(soa)) + comp)
    assert dump(tmp_path / "lzf.pcd") == ref
    # PLY
    ply_hdr = lambda fmt: (f"ply\nformat {fmt} 1.0\ncomment test\nelement vertex 300\nproperty float x\nproperty float y\nproperty float z\n"
                           "property float nx\nproperty float ny\nproperty float nz\nproperty uchar red\nelement face 0\n"
                           "property list uchar int vertex_indices\nend_header\n")
    with open(tmp_path / "a.ply", "w") as f:
        f.write(ply_hdr("ascii"))
        for p, q in zip(xyz, nrm):
            f.write(" ".join(repr(float(v)) for v in list(p) + list(q)) + " 7\n")
    with open(tmp_path / "b.ply", "wb") as f:
        f.write(ply_hdr("binary_little_endian").encode())
        for p, q in zip(xyz, nrm):
            f.write(struct.pack("<6fB", *p, *q, 7))
    assert dump(tmp_path / "a.ply") == ref and dump(tmp_path / "b.ply") == ref
    # corrupt compressed payload is rejected, not mis-read
    open(tmp_path / "bad.pcd", "wb").write(hdr.encode() + struct.pack("<II", len(comp), len(soa)) + comp[:-5] + b"\xff" * 5)
    assert dump(tmp_path / "bad.pcd")[0] == 0


def test_cfg_parser_against_the_references_own_parser(cli, tmp_path, golden_dir):
    """The shim's util::ConfigFile, HandGeometry(filepath) and ImageGeometry(filepath) against the REFERENCE's (its
    config_file.cpp, hand_geometry.cpp and image_geometry.cpp, the sources of the reference that build without PCL / Eigen /
    OpenCV; their answers are stored in tests/golden/ref_config_parser.json): identical values for every key and getter on a
    cfg with the format's corner cases and on the shipped cfg files."""
    import ctypes as C
    with open(os.path.join(golden_dir, "ref_config_parser.json")) as f:
        ref = json.load(f)
    got = config_parser_answers(C.CDLL(os.path.join(HOST, "libgpd_host.so")), False, os.path.join(golden_dir, "cfg"), str(tmp_path))
    assert sorted(got) == sorted(ref)
    for k in ref:
        assert got[k] == ref[k], (k, ref[k], got[k])
    assert got["does_not_exist.cfg|alpha"][0] == 0


def _write_detector_cfg(tmp_path, w, extra=""):
    os.makedirs(tmp_path / "params", exist_ok=True)
    names = ["conv1_weights", "conv1_biases", "conv2_weights", "conv2_biases", "ip1_weights", "ip1_biases", "ip2_weights", "ip2_biases"]
    for n, a in zip(names, w):
        a.astype(np.float32).tofile(tmp_path / "params" / (n + ".bin"))
    (tmp_path / "main.cfg").write_text(f"hand_geometry_filename = 0\nimage_geometry_filename = 0\nweights_file = {tmp_path}/params/\n"
                                       "image_num_channels = 15\nvoxelize = 0\n" + extra)
    return str(tmp_path / "main.cfg")


@pytest.mark.gpu
def test_sequential_importance_sampling_cli_matches_the_oracle(cli, tmp_path):
    """cem_detect_grasps (SequentialImportanceSampling::detectGrasps, sequential_importance_sampling.cpp:54-185) through the
    shim: hand search at arbitrary sample positions on the device for every round (gpdb_set_samples), classification at
    the end. The CLI prints the positions of the hand sets it kept; the oracle recomputes hands and scores AT those positions
    (Cloud::setSamples) — the grasps must be the same set with the same scores, and every kept position must carry a hand."""
    from conftest import load_weights
    from gpd_b200 import abi
    from oracle import oracle
    k = scenes.krylon_cloud()
    write_pcd(tmp_path / "krylon.pcd", k["xyz"], k["normals"], binary=True)
    w, _ = load_weights(15)
    cfg = _write_detector_cfg(tmp_path, w, "num_samples = 100\nnum_init_samples = 40\nnum_iterations = 3\n"
                              "num_samples_per_iteration = 60\nprob_rand_samples = 0.25\nstandard_deviation = 0.01\n"
                              "min_score = -1000000\nmin_inliers = 0\nnum_selected = 1000\n")
    out = subprocess.check_output([cli, cfg, str(tmp_path / "krylon.pcd"), "--sis", "7"]).decode()
    pos = np.array([[float(x) for x in l.split()[1:]] for l in out.splitlines() if l.startswith("SIS_SAMPLE")])
    grasps = np.array([[float(x) for x in l.split()[1:]] for l in out.splitlines() if l.startswith("SIS_GRASP")])
    res = [l for l in out.splitlines() if l.startswith("RESULT")][0]
    assert int(res.split("evaluated=")[1].split()[0]) == 40 + 3 * 60
    assert len(pos) == int(res.split("hand_sets=")[1]) and len(pos) >= 10 and len(grasps) == int(res.split("n_grasps=")[1].split()[0])
    # off-cloud positions were evaluated (Gaussian draws), not only cloud points
    d = np.abs(pos[:, None, :].astype(np.float32) - k["xyz"][None, :, :]).sum(2).min(1)
    assert np.count_nonzero(d > 1e-6) >= 5
    oc = oracle.OracleCloud(k["xyz"], k["normals"], k["cam_source"], k["view_points"])
    p = abi.default_params(15)
    ro = oc.detect(p, oracle.WeightPack(w), oc.set_samples(pos))
    co = ro["candidates"]
    assert len(np.unique(co["sample_slot"])) == len(pos)  # every kept position carries at least one hand
    assert len(co) == len(grasps)
    assert np.allclose(co["position"], grasps[:, 1:4], atol=1e-9, rtol=0)
    assert np.abs(co["score"] - grasps[:, 0]).max() <= 1e-4 * np.abs(co["score"]).max()
    # seeded: the same seed reproduces the run, another seed explores other positions
    again = subprocess.check_output([cli, cfg, str(tmp_path / "krylon.pcd"), "--sis", "7"]).decode()
    assert [l for l in again.splitlines() if l.startswith("SIS_")] == [l for l in out.splitlines() if l.startswith("SIS_")]
    other = subprocess.check_output([cli, cfg, str(tmp_path / "krylon.pcd"), "--sis", "8"]).decode()
    assert [l for l in other.splitlines() if l.startswith("SIS_SAMPLE")] != [l for l in out.splitlines() if l.startswith("SIS_SAMPLE")]


@pytest.mark.gpu
def test_detect_grasps_cli_on_two_gpus_equals_one(cli, tmp_path):
    """detect_grasps --gpus 2: GraspDetector::detectGraspsMultiGpu (one thread + context per device, gpdb_comm_init /
    gpdb_set_cloud_bcast / gpdb_detect_sharded inside the library) returns the same selected grasps as the single-GPU run."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from conftest import load_weights
    k = scenes.krylon_cloud()
    write_pcd(tmp_path / "krylon.pcd", k["xyz"], k["normals"], binary=True)
    w, _ = load_weights(15)
    cfg = _write_detector_cfg(tmp_path, w, "num_samples = 1500\nmin_inliers = 0\nnum_selected = 25\n")
    one = subprocess.check_output([cli, cfg, str(tmp_path / "krylon.pcd")]).decode()
    two = subprocess.check_output([cli, cfg, str(tmp_path / "krylon.pcd"), "--gpus", "2"]).decode()
    pick = lambda o: [l for l in o.splitlines() if l.startswith("RESULT") or l.startswith("--- grasp") or "position" in l.lower() or "score" in l.lower()]
    r1 = [l for l in one.splitlines() if l.startswith("RESULT")][0]
    r2 = [l for l in two.splitlines() if l.startswith("RESULT")][0]
    assert r1 == r2, (r1, r2)
    c1 = [l for l in one.splitlines() if "gripper width" in l][0].split(":")[1].split()[0]
    c2 = [l for l in two.splitlines() if "gripper width" in l][0].split(":")[1].split()[0]
    assert c1 == c2


@pytest.mark.gpu
def test_device_clustering_equals_the_host_restatement(cli):
    """gpdb_find_clusters (one warp per hand, inliers folded in index order) against the shim's host Clustering::findClusters
    (itself checked against a Python restatement above): bit-equal cluster records on real detections."""
    import ctypes as C
    from conftest import load_weights
    from gpd_b200 import abi, lib
    k = scenes.krylon_cloud()
    w, _ = load_weights(15)
    p = lib.default_params(channels=15)
    ctx = lib.Context(p)
    ctx.set_weights(w)
    ctx.set_cloud(k["xyz"], k["normals"], k["cam_source"], k["view_points"])
    hands = ctx.detect_select(np.arange(0, len(k["xyz"]), 2, dtype=np.int32), 400)["candidates"]
    assert len(hands) == 400
    H = C.CDLL(os.path.join(HOST, "libgpd_host.so"))
    H.gpdFindClusters.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    for min_inliers in (1, 3, 10):
        ref = np.zeros(len(hands), dtype=abi.POSE_DTYPE)
        n = H.gpdFindClusters(hands.ctypes.data, len(hands), min_inliers, 0, ref.ctypes.data)
        dev = ctx.find_clusters(hands, min_inliers)
        assert len(dev) == n and n > 0
        for f in ("position", "score", "frame", "sample_index", "pose_slot", "full_antipodal"):
            assert np.array_equal(dev[f], ref[:n][f]), (min_inliers, f)
    assert len(ctx.find_clusters(hands[:1], 1)) == 0 and len(ctx.find_clusters(hands[:0], 1)) == 0
    ctx.close()
