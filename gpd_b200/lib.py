"""ctypes binding of libgpd_b200.so — the CUDA product library (include/gpd_b200.h).

The library is built in-tree (gpd_b200/csrc/Makefile, __graft_entry__.build()). There is no CPU
fallback: if the shared object is missing this module raises, and every compute call returns
GPDB_ERR_CUDA when no sm_100 device is present.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# GPD_B200_LIB overrides the library path (A/B comparison of builds during development); default: the in-tree build
SO_PATH = os.environ.get("GPD_B200_LIB") or os.path.join(_HERE, "libgpd_b200.so")
_LIB = None

EXPORTS = [
    "gpdb_params_default", "gpdb_create", "gpdb_destroy", "gpdb_last_error", "gpdb_load_weights_dir",
    "gpdb_set_weights", "gpdb_set_cloud", "gpdb_detect", "gpdb_frames", "gpdb_hand_search", "gpdb_images",
    "gpdb_classify", "gpdb_free_result", "gpdb_last_timings", "gpdb_build_info", "gpdb_detect_resident",
    "gpdb_set_stream", "gpdb_debug_phase_cycles", "gpdb_preprocess_params_default", "gpdb_preprocess",
    "gpdb_get_cloud", "gpdb_get_cloud_source_index", "gpdb_preprocess_timings", "gpdb_detect_select", "gpdb_load_weights_file", "gpdb_read_weights_file", "gpdb_set_samples",
    "gpdb_comm_unique_id", "gpdb_comm_init", "gpdb_comm_destroy", "gpdb_shard_bounds", "gpdb_set_cloud_bcast",
    "gpdb_detect_sharded", "gpdb_detect_sharded_resident", "gpdb_slot_bytes", "gpdb_find_clusters", "gpdb_reevaluate", "gpdb_set_overlap",
    "gpdb_plane_params_default", "gpdb_sample_above_plane",
]


class GpdbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{code}] {msg}")
        self.code = code


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). gpd_b200 has no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp = C.c_void_p
    L.gpdb_params_default.argtypes = [C.POINTER(abi.Params)]
    L.gpdb_create.argtypes = [C.POINTER(abi.Params), C.POINTER(vp)]
    L.gpdb_destroy.argtypes = [vp]
    L.gpdb_last_error.restype = C.c_char_p
    L.gpdb_last_error.argtypes = [vp]
    L.gpdb_load_weights_dir.argtypes = [vp, C.c_char_p]
    L.gpdb_set_weights.argtypes = [vp] + [vp] * 8
    L.gpdb_load_weights_file.argtypes = [vp, C.c_char_p, C.c_char_p]
    L.gpdb_read_weights_file.argtypes = [C.c_char_p, C.c_char_p, C.c_int32, vp, vp, C.c_char_p, C.c_int32]
    L.gpdb_set_cloud.argtypes = [vp, vp, vp, vp, C.c_int32, vp, C.c_int32]
    L.gpdb_detect.argtypes = [vp, vp, C.c_int32, C.POINTER(abi.Result)]
    L.gpdb_hand_search.argtypes = [vp, vp, C.c_int32, C.POINTER(abi.Result)]
    L.gpdb_detect_select.argtypes = [vp, vp, C.c_int32, C.c_int32, C.POINTER(abi.Result)]
    L.gpdb_frames.argtypes = [vp, vp, C.c_int32, vp, vp]
    L.gpdb_images.argtypes = [vp, vp, C.c_int32, vp]
    L.gpdb_classify.argtypes = [vp, vp, C.c_int32, vp, vp]
    L.gpdb_free_result.argtypes = [C.POINTER(abi.Result)]
    L.gpdb_last_timings.argtypes = [vp, vp]
    L.gpdb_build_info.restype = C.c_char_p
    L.gpdb_detect_resident.argtypes = [vp, vp, C.c_int32, vp, vp, C.POINTER(abi.Result)]
    L.gpdb_set_stream.argtypes = [vp, vp]
    L.gpdb_debug_phase_cycles.argtypes = [vp, C.c_int, vp]
    L.gpdb_preprocess_params_default.argtypes = [C.POINTER(abi.PreprocessParams)]
    L.gpdb_preprocess.argtypes = [vp, vp, vp, vp, C.c_int32, vp, C.c_int32, C.POINTER(abi.PreprocessParams)]
    L.gpdb_get_cloud.argtypes = [vp, vp, vp, vp]
    L.gpdb_set_samples.argtypes = [vp, vp, C.c_int32]
    L.gpdb_get_cloud_source_index.argtypes = [vp, vp]
    L.gpdb_preprocess_timings.argtypes = [vp, vp]
    L.gpdb_comm_unique_id.argtypes = [vp]
    L.gpdb_comm_init.argtypes = [vp, vp, C.c_int32, C.c_int32]
    L.gpdb_comm_destroy.argtypes = [vp]
    L.gpdb_shard_bounds.argtypes = [C.c_int32, C.c_int32, C.c_int32, vp, vp, vp]
    L.gpdb_shard_bounds.restype = None
    L.gpdb_set_cloud_bcast.argtypes = [vp, C.c_int32, vp, vp, vp, C.c_int32, vp, C.c_int32]
    L.gpdb_detect_sharded.argtypes = [vp, vp, C.c_int32, C.POINTER(abi.Result)]
    L.gpdb_detect_sharded_resident.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, C.POINTER(abi.Result)]
    L.gpdb_slot_bytes.argtypes = [C.c_int32, C.c_int32]
    L.gpdb_slot_bytes.restype = C.c_int64
    L.gpdb_find_clusters.argtypes = [vp, vp, C.c_int32, C.c_int32, vp]
    L.gpdb_reevaluate.argtypes = [vp, vp, C.c_int32, vp]
    L.gpdb_set_overlap.argtypes = [vp, C.c_int32]
    L.gpdb_plane_params_default.argtypes = [C.POINTER(abi.PlaneParams)]
    L.gpdb_plane_params_default.restype = None
    L.gpdb_sample_above_plane.argtypes = [vp, C.POINTER(abi.PlaneParams), vp, C.POINTER(abi.PlaneInfo)]
    _LIB = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def default_params(**over):
    p = abi.Params()
    lib().gpdb_params_default(C.byref(p))
    q = abi.default_params(p.image_num_channels)
    for name, _ in abi.Params._fields_:  # the two defaults must agree (tests check it)
        pass
    chan = over.pop("channels", None)
    if chan is not None:
        p.image_num_channels = chan
    for k, v in over.items():
        if k == "hand_axes":
            p.num_hand_axes = len(v)
            for i, a in enumerate(v):
                p.hand_axes[i] = a
        elif k in ("workspace_grasps", "direction"):
            for i, a in enumerate(v):
                getattr(p, k)[i] = a
        else:
            setattr(p, k, v)
    del q
    return p


def preprocess_params(**over):
    """gpdb_preprocess_params with the reference defaults (cfg/eigen_params.cfg:16-21), overridden by keyword."""
    p = abi.PreprocessParams()
    lib().gpdb_preprocess_params_default(C.byref(p))
    for k, v in over.items():
        if k == "workspace":
            p.workspace[:] = list(v)
        else:
            setattr(p, k, v)
    return p


def plane_params(**over):
    """gpdb_plane_params with the library defaults (threshold 0.01, 1024 hypotheses, seed 1), overridden by keyword."""
    p = abi.PlaneParams()
    lib().gpdb_plane_params_default(C.byref(p))
    for k, v in over.items():
        setattr(p, k, v)
    return p


def read_weights_file(weights_file, channels, model_file=None):
    """Host-side import of a .caffemodel or an OpenVINO IR into the eight arrays of the .bin layout (no device needed).
    Returns (arrays, relu_layers)."""
    sizes = [20 * channels * 25, 20, 50 * 20 * 25, 50, 500 * 7200, 500, 1000, 2]
    arrs = [np.zeros(s, np.float32) for s in sizes]
    ptrs = (C.c_void_p * 8)(*[a.ctypes.data for a in arrs])
    relu = C.c_int32(-1)
    err = C.create_string_buffer(512)
    rc = lib().gpdb_read_weights_file(None if model_file is None else model_file.encode(), weights_file.encode(), channels, ptrs,
                                      C.byref(relu), err, 512)
    if rc != 0:
        raise GpdbError(rc, err.value.decode())
    return arrs, relu.value


class Context:
    """One gpdb_ctx: one CUDA device + stream (gpdb_create ... gpdb_destroy)."""

    def __init__(self, params):
        self.params = params
        self.h = C.c_void_p()
        rc = lib().gpdb_create(C.byref(params), C.byref(self.h))
        if rc != 0:
            self.h = None
            raise GpdbError(rc, lib().gpdb_last_error(None).decode())
        self._keep = []

    def close(self):
        if getattr(self, "h", None):
            lib().gpdb_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _check(self, rc):
        if rc < 0:
            raise GpdbError(rc, lib().gpdb_last_error(self.h).decode())
        return rc

    def load_weights_dir(self, d):
        if not d.endswith("/"):
            d += "/"
        self._check(lib().gpdb_load_weights_dir(self.h, d.encode()))

    def load_weights_file(self, weights_file, model_file=None):
        """.bin directory, .caffemodel or OpenVINO IR (.bin + .xml), as Classifier::create's weights_file / model_file."""
        self._check(lib().gpdb_load_weights_file(self.h, None if model_file is None else model_file.encode(), weights_file.encode()))

    def set_weights(self, arrays):
        arrs = [np.ascontiguousarray(a, dtype=np.float32).ravel() for a in arrays]
        self._check(lib().gpdb_set_weights(self.h, *[_p(a) for a in arrs]))

    def set_cloud(self, xyz, normals, cam_source=None, view_points=None):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        normals = np.ascontiguousarray(normals, dtype=np.float64)
        vp = np.ascontiguousarray(view_points if view_points is not None else np.zeros((1, 3)), dtype=np.float64)
        cam = None if cam_source is None else np.ascontiguousarray(cam_source, dtype=np.int32)
        self._check(lib().gpdb_set_cloud(self.h, _p(xyz), _p(normals), _p(cam), xyz.shape[0], _p(vp), vp.shape[0]))

    def preprocess(self, xyz, cam_source=None, view_points=None, pp=None, normals=None, read_back=True):
        """CandidatesGenerator::preprocessPointCloud on the device (gpdb_preprocess): NaN / workspace filter,
        voxelisation, normal estimation; installs the processed cloud. Returns the processed cloud as a dict
        (xyz, normals, cam_source, view_points, src) or just N' when read_back is False."""
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        vp = np.ascontiguousarray(view_points if view_points is not None else np.zeros((1, 3)), dtype=np.float64)
        cam = None if cam_source is None else np.ascontiguousarray(cam_source, dtype=np.int32)
        nrm = None if normals is None else np.ascontiguousarray(normals, dtype=np.float64)
        if pp is None:
            pp = preprocess_params()
        n = self._check(lib().gpdb_preprocess(self.h, _p(xyz), _p(nrm), _p(cam), xyz.shape[0], _p(vp), vp.shape[0],
                                              C.byref(pp)))
        if not read_back:
            return n
        out = self.get_cloud() if n > 0 else {"xyz": np.zeros((0, 3), np.float32), "normals": np.zeros((0, 3)),
                                              "cam_source": np.zeros((0, vp.shape[0]), np.int32)}
        out["view_points"] = vp
        if n > 0:
            src = np.zeros(n, np.int32)
            self._check(lib().gpdb_get_cloud_source_index(self.h, _p(src)))
            out["src"] = src
        else:
            out["src"] = np.zeros(0, np.int32)
        return out

    def sample_above_plane(self, pp=None):
        """Cloud::sampleAbovePlane on the installed cloud (gpdb_sample_above_plane): (off-plane indices ascending, info
        dict). An empty index array means the plane fit failed and the whole cloud stays sampled."""
        if pp is None:
            pp = plane_params()
        n_pts = self._check(lib().gpdb_get_cloud(self.h, None, None, None))
        idx = np.zeros(max(n_pts, 1), np.int32)
        info = abi.PlaneInfo()
        n = self._check(lib().gpdb_sample_above_plane(self.h, C.byref(pp), _p(idx), C.byref(info)))
        return idx[:n].copy(), abi.plane_info_to_dict(info)

    # ---- multi-GPU sharding inside the boundary (gpdb_comm_*, SURVEY.md 8(e)) ----
    def comm_init(self, unique_id, rank, nranks):
        """ncclCommInitRank on this context's device; unique_id = 128 bytes from comm_unique_id() of one rank."""
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(lib().gpdb_comm_init(self.h, buf, int(rank), int(nranks)))
        self.rank, self.nranks = int(rank), int(nranks)

    def set_cloud_bcast(self, root, xyz=None, normals=None, cam_source=None, view_points=None):
        """gpdb_set_cloud on every rank from the root's host arrays (ncclBroadcast of the device copies)."""
        if xyz is None:
            return self._check(lib().gpdb_set_cloud_bcast(self.h, int(root), None, None, None, 0, None, 0))
        xyz = np.ascontiguousarray(xyz, dtype=np.float32)
        normals = np.ascontiguousarray(normals, dtype=np.float64)
        vp = np.ascontiguousarray(view_points if view_points is not None else np.zeros((1, 3)), dtype=np.float64)
        cam = None if cam_source is None else np.ascontiguousarray(cam_source, dtype=np.int32)
        return self._check(lib().gpdb_set_cloud_bcast(self.h, int(root), _p(xyz), _p(normals), _p(cam), xyz.shape[0], _p(vp), vp.shape[0]))

    def detect_sharded(self, sample_idx):
        """gpdb_detect over sharded samples: gathered pose_flags / pose_scores of all ranks + this rank's pose records."""
        sidx = np.ascontiguousarray(sample_idx, dtype=np.int32)
        res = abi.Result()
        self._check(lib().gpdb_detect_sharded(self.h, _p(sidx), len(sidx), C.byref(res)))
        n, P, nc = res.n_samples, res.poses_per_sample, res.n_candidates
        out = {"pose_flags": np.ctypeslib.as_array(res.pose_flags, (n, P)).copy(),
               "pose_scores": np.ctypeslib.as_array(res.pose_scores, (n, P)).copy(),
               "n_candidates": nc, "n_total_candidates": res.n_total_candidates,
               "candidates": np.frombuffer(C.string_at(res.candidates, nc * C.sizeof(abi.Pose)), dtype=abi.POSE_DTYPE).copy()
               if nc else np.zeros(0, dtype=abi.POSE_DTYPE)}
        lib().gpdb_free_result(C.byref(res))
        return out

    def detect_sharded_raw(self, sidx_i32, res):
        return self._check(lib().gpdb_detect_sharded(self.h, _p(sidx_i32), len(sidx_i32), C.byref(res)))

    def detect_sharded_resident(self, d_sidx_local_ptr, n_local, slot_samples, d_gathered_ptr, stats):
        return self._check(lib().gpdb_detect_sharded_resident(self.h, C.c_void_p(d_sidx_local_ptr), int(n_local), int(slot_samples),
                                                              C.c_void_p(d_gathered_ptr), C.byref(stats)))

    def reevaluate(self, hands):
        """HandSearch::reevaluateHypotheses against the installed cloud: (labels int32, re-labelled records)."""
        hands = np.array(hands, dtype=abi.POSE_DTYPE, copy=True)
        labels = np.zeros(len(hands), np.int32)
        self._check(lib().gpdb_reevaluate(self.h, _p(hands), len(hands), _p(labels)))
        return labels, hands

    def find_clusters(self, hands, min_inliers):
        """Clustering::findClusters (remove_inliers = false) on the device; hands / result: abi.POSE_DTYPE records."""
        hands = np.ascontiguousarray(hands, dtype=abi.POSE_DTYPE)
        out = np.zeros(len(hands), dtype=abi.POSE_DTYPE)
        n = self._check(lib().gpdb_find_clusters(self.h, _p(hands), len(hands), int(min_inliers), _p(out)))
        return out[:n].copy()

    def set_samples(self, samples):
        """Cloud::setSamples: arbitrary float64 positions [n, 3]; returns the sample indices that address them."""
        sm = np.ascontiguousarray(samples, dtype=np.float64)
        first = self._check(lib().gpdb_set_samples(self.h, _p(sm), len(sm)))
        return np.arange(first, first + len(sm), dtype=np.int32)

    def get_cloud(self):
        n = self._check(lib().gpdb_get_cloud(self.h, None, None, None))
        xyz = np.zeros((n, 3), np.float32)
        nrm = np.zeros((n, 3), np.float64)
        self._check(lib().gpdb_get_cloud(self.h, _p(xyz), _p(nrm), None))
        return {"xyz": xyz, "normals": nrm, "cam_source": self._cam_source(n)}

    def _cam_source(self, n, kmax=8):
        # the camera count is not exported separately: read k x N into a buffer sized for GPDB_MAX_CAMERAS
        buf = np.full(n * kmax, -1, np.int32)
        self._check(lib().gpdb_get_cloud(self.h, None, None, _p(buf)))
        k = int(np.count_nonzero(buf >= 0)) // max(n, 1)
        return buf[: n * k].reshape(n, k).copy()

    def preprocess_timings(self):
        ms = np.zeros(6)
        lib().gpdb_preprocess_timings(self.h, _p(ms))
        return ms

    def _result(self, fn, sample_idx):
        sidx = np.ascontiguousarray(sample_idx, dtype=np.int32)
        res = abi.Result()
        self._check(fn(self.h, _p(sidx), len(sidx), C.byref(res)))
        S, Cc = self.params.image_size, self.params.image_num_channels
        out = abi.result_to_numpy(res, S * S * Cc)
        lib().gpdb_free_result(C.byref(res))
        return out

    def detect(self, sample_idx):
        return self._result(lib().gpdb_detect, sample_idx)

    def detect_select(self, sample_idx, num_selected):
        """detectGrasps + selectGrasps: the num_selected best candidates, sorted on the device (gpdb_detect_select)."""
        sidx = np.ascontiguousarray(sample_idx, dtype=np.int32)
        res = abi.Result()
        self._check(lib().gpdb_detect_select(self.h, _p(sidx), len(sidx), int(num_selected), C.byref(res)))
        S, Cc = self.params.image_size, self.params.image_num_channels
        out = abi.result_to_numpy(res, S * S * Cc)
        lib().gpdb_free_result(C.byref(res))
        return out

    def detect_select_raw(self, sidx_i32, num_selected, res):
        """Timed path for bench.py; caller frees `res`."""
        return self._check(lib().gpdb_detect_select(self.h, _p(sidx_i32), len(sidx_i32), int(num_selected), C.byref(res)))

    def detect_raw(self, sidx_i32, res):
        """Timed path for bench.py: no numpy conversion; caller frees `res`."""
        return self._check(lib().gpdb_detect(self.h, _p(sidx_i32), len(sidx_i32), C.byref(res)))

    def detect_resident(self, d_sidx_ptr, n, d_flags_ptr, d_scores_ptr, stats):
        """Device-resident path (raw device pointers as ints); returns n_candidates."""
        return self._check(lib().gpdb_detect_resident(self.h, C.c_void_p(d_sidx_ptr), n, C.c_void_p(d_flags_ptr),
                                                      C.c_void_p(d_scores_ptr), C.byref(stats)))

    def set_overlap(self, enable):
        """Hand search of the chunks ahead on its own stream (default on); off = one stream, exclusive stage timers."""
        self._check(lib().gpdb_set_overlap(self.h, int(bool(enable))))

    def set_stream(self, cuda_stream_ptr):
        self._check(lib().gpdb_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def hand_search(self, sample_idx):
        return self._result(lib().gpdb_hand_search, sample_idx)

    def frames(self, sample_idx):
        sidx = np.ascontiguousarray(sample_idx, dtype=np.int32)
        n = len(sidx)
        frames = np.zeros((n, 9))
        valid = np.zeros(n, np.uint8)
        self._check(lib().gpdb_frames(self.h, _p(sidx), n, _p(frames), _p(valid)))
        return frames, valid

    def images(self, poses):
        poses = np.ascontiguousarray(poses, dtype=abi.POSE_DTYPE)
        n = len(poses)
        S, Cc = self.params.image_size, self.params.image_num_channels
        out = np.zeros((n, S, S, Cc), np.uint8)
        self._check(lib().gpdb_images(self.h, _p(poses), n, _p(out)))
        return out

    def classify(self, images):
        images = np.ascontiguousarray(images, dtype=np.uint8)
        n = images.shape[0]
        scores = np.zeros(n, np.float32)
        logits = np.zeros((n, 2), np.float32)
        self._check(lib().gpdb_classify(self.h, _p(images), n, _p(scores), _p(logits)))
        return scores, logits

    def phase_cycles(self, enable=1):
        out = np.zeros(16, np.uint64)
        self._check(lib().gpdb_debug_phase_cycles(self.h, enable, _p(out)))
        return out

    def last_timings(self):
        ms = np.zeros(8)
        lib().gpdb_last_timings(self.h, _p(ms))
        return ms


def comm_unique_id():
    """ncclGetUniqueId (128 bytes): call on one rank and distribute to the others."""
    buf = C.create_string_buffer(128)
    rc = lib().gpdb_comm_unique_id(buf)
    if rc != 0:
        raise GpdbError(rc, lib().gpdb_last_error(None).decode())
    return buf.raw


def shard_bounds(n, rank, nranks):
    """(lo, hi, slot_samples) of gpdb_shard_bounds: the slice of `rank` and the fixed slot size of the all-gather."""
    lo, hi, st = C.c_int32(), C.c_int32(), C.c_int32()
    lib().gpdb_shard_bounds(int(n), int(rank), int(nranks), C.byref(lo), C.byref(hi), C.byref(st))
    return lo.value, hi.value, st.value


def slot_bytes(slot_samples, P):
    return int(lib().gpdb_slot_bytes(int(slot_samples), int(P)))


def free_result(res):
    lib().gpdb_free_result(C.byref(res))
