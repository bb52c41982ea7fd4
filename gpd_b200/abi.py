"""ctypes mirror of include/gpd_b200.h (the C-ABI types of the grasp-candidate hot path).

Only type definitions live here; they are shared by the product loader (gpd_b200/lib.py) and by
the test-only oracle loader (oracle/oracle.py) because both speak the same boundary structs.
"""
import ctypes as C

import numpy as np

MAX_HAND_AXES = 3
POSE_VALID, POSE_FILTERED, POSE_HALF, POSE_FULL = 1, 2, 4, 8


class Params(C.Structure):
    """gpdb_params — field names are the reference's cfg keys (grasp_detector.cpp:48-185)."""

    _fields_ = [
        ("finger_width", C.c_double),
        ("hand_outer_diameter", C.c_double),
        ("hand_depth", C.c_double),
        ("hand_height", C.c_double),
        ("init_bite", C.c_double),
        ("volume_width", C.c_double),
        ("volume_depth", C.c_double),
        ("volume_height", C.c_double),
        ("image_size", C.c_int32),
        ("image_num_channels", C.c_int32),
        ("nn_radius", C.c_double),
        ("num_orientations", C.c_int32),
        ("num_finger_placements", C.c_int32),
        ("num_hand_axes", C.c_int32),
        ("hand_axes", C.c_int32 * MAX_HAND_AXES),
        ("deepen_hand", C.c_int32),
        ("friction_coeff", C.c_double),
        ("min_viable", C.c_int32),
        ("min_aperture", C.c_double),
        ("max_aperture", C.c_double),
        ("workspace_grasps", C.c_double * 6),
        ("filter_approach_direction", C.c_int32),
        ("direction", C.c_double * 3),
        ("thresh_rad", C.c_double),
        ("batch_size", C.c_int32),
        ("relu_after_conv", C.c_int32),
        ("shadow_mode", C.c_int32),
        ("device", C.c_int32),
        ("chunk_samples", C.c_int32),
        ("keep_images", C.c_int32),
        ("lenet_impl", C.c_int32),
    ]


class Pose(C.Structure):
    """gpdb_pose = candidate::Hand (include/gpd/candidate/hand.h:267-276)."""

    _fields_ = [
        ("sample", C.c_double * 3),
        ("frame", C.c_double * 9),
        ("position", C.c_double * 3),
        ("top", C.c_double),
        ("bottom", C.c_double),
        ("center", C.c_double),
        ("width", C.c_double),
        ("score", C.c_float),
        ("sample_index", C.c_int32),
        ("sample_slot", C.c_int32),
        ("pose_slot", C.c_int16),
        ("finger_idx", C.c_int16),
        ("half_antipodal", C.c_uint8),
        ("full_antipodal", C.c_uint8),
        ("pad_", C.c_uint8 * 6),
    ]


POSE_DTYPE = np.dtype(
    [
        ("sample", "<f8", (3,)),
        ("frame", "<f8", (9,)),
        ("position", "<f8", (3,)),
        ("top", "<f8"),
        ("bottom", "<f8"),
        ("center", "<f8"),
        ("width", "<f8"),
        ("score", "<f4"),
        ("sample_index", "<i4"),
        ("sample_slot", "<i4"),
        ("pose_slot", "<i2"),
        ("finger_idx", "<i2"),
        ("half_antipodal", "u1"),
        ("full_antipodal", "u1"),
        ("pad_", "u1", (6,)),
    ],
    align=True,
)
assert POSE_DTYPE.itemsize == C.sizeof(Pose), (POSE_DTYPE.itemsize, C.sizeof(Pose))


class Result(C.Structure):
    """gpdb_result — callee-allocated SoA result."""

    _fields_ = [
        ("n_samples", C.c_int32),
        ("poses_per_sample", C.c_int32),
        ("frame_valid", C.POINTER(C.c_uint8)),
        ("frames", C.POINTER(C.c_double)),
        ("pose_flags", C.POINTER(C.c_uint8)),
        ("pose_scores", C.POINTER(C.c_float)),
        ("n_candidates", C.c_int32),
        ("candidates", C.POINTER(Pose)),
        ("images", C.POINTER(C.c_uint8)),
        ("ms_candidates", C.c_double),
        ("ms_images", C.c_double),
        ("ms_classify", C.c_double),
        ("kernel_launches", C.c_int64),
        ("n_total_candidates", C.c_int32),
        ("owner_", C.c_void_p),
    ]


class PreprocessParams(C.Structure):
    """gpdb_preprocess_params — cfg keys of CandidatesGenerator::preprocessPointCloud
    (candidates_generator.cpp:14-37, grasp_detector.cpp:50-66)."""

    _fields_ = [
        ("workspace", C.c_double * 6),
        ("voxel_size", C.c_double),
        ("normals_radius", C.c_double),
        ("voxelize", C.c_int32),
        ("estimate_normals", C.c_int32),
    ]


def default_preprocess_params(**over):
    """Reference defaults (cfg/eigen_params.cfg:16-21, grasp_detector.cpp:56-66)."""
    p = PreprocessParams()
    p.workspace[:] = [-1.0, 1.0, -1.0, 1.0, -1.0, 1.0]
    p.voxel_size = 0.003
    p.normals_radius = 0.03
    p.voxelize = 1
    p.estimate_normals = 1
    for k, v in over.items():
        if k == "workspace":
            p.workspace[:] = list(v)
        else:
            setattr(p, k, v)
    return p


class PlaneParams(C.Structure):
    """gpdb_plane_params — the support-plane fit of sample_above_plane (include/gpd_b200_plane.h)."""

    _fields_ = [
        ("distance_threshold", C.c_double),
        ("num_hypotheses", C.c_int32),
        ("seed", C.c_uint64),
    ]


class PlaneInfo(C.Structure):
    """gpdb_plane_info — what the plane fit found."""

    _fields_ = [
        ("coefficients", C.c_float * 4),
        ("hypothesis_coefficients", C.c_float * 4),
        ("hypothesis", C.c_int32),
        ("hypothesis_inliers", C.c_int32),
        ("inliers", C.c_int32),
        ("refined", C.c_int32),
    ]


def default_plane_params(**over):
    """Defaults of gpdb_plane_params_default: threshold 0.01 (cloud.cpp:418), 1024 hypotheses, seed 1."""
    p = PlaneParams(0.01, 1024, 1)
    for k, v in over.items():
        setattr(p, k, v)
    return p


def plane_info_to_dict(info):
    return {"coefficients": np.array(info.coefficients[:], np.float32),
            "hypothesis_coefficients": np.array(info.hypothesis_coefficients[:], np.float32),
            "hypothesis": info.hypothesis, "hypothesis_inliers": info.hypothesis_inliers, "inliers": info.inliers,
            "refined": info.refined}


def default_params(channels=15, **over):
    """The reference defaults (gpdb_params_default in C), restated for the oracle loader.

    cfg/hand_geometry.cfg:8-12, cfg/image_geometry_15channels.cfg:8-12, cfg/eigen_params.cfg:36-42,
    grasp_detector.cpp:158-174.
    """
    p = Params()
    p.finger_width, p.hand_outer_diameter, p.hand_depth = 0.01, 0.12, 0.06
    p.hand_height, p.init_bite = 0.02, 0.01
    p.volume_width, p.volume_depth, p.volume_height = 0.10, 0.06, 0.02
    p.image_size, p.image_num_channels = 60, channels
    p.nn_radius = 0.01
    p.num_orientations, p.num_finger_placements = 8, 10
    p.num_hand_axes = 1
    p.hand_axes[0] = 2
    p.deepen_hand = 1
    p.friction_coeff, p.min_viable = 20.0, 6
    p.min_aperture, p.max_aperture = 0.0, 0.085
    for i, v in enumerate([-1, 1, -1, 1, -1, 1]):
        p.workspace_grasps[i] = v
    p.filter_approach_direction = 0
    p.direction[0], p.direction[1], p.direction[2] = 1.0, 0.0, 0.0
    p.thresh_rad = 2.3
    p.batch_size = 0
    p.relu_after_conv = 0
    p.shadow_mode = 0
    p.device = 0
    p.chunk_samples = 0
    p.keep_images = 0
    p.lenet_impl = 0
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
    return p


def result_to_numpy(res, image_bytes):
    """Copy a gpdb_result into numpy arrays (so the C result can be freed)."""
    n, P = res.n_samples, res.poses_per_sample
    nc = res.n_candidates
    full = bool(res.frames)  # gpdb_detect_select returns the selected pose records only
    out = {
        "n_samples": n,
        "poses_per_sample": P,
        "frame_valid": None if not full else np.ctypeslib.as_array(res.frame_valid, (n,)).copy() if n else np.zeros(0, np.uint8),
        "frames": None if not full else np.ctypeslib.as_array(res.frames, (n, 9)).copy() if n else np.zeros((0, 9)),
        "pose_flags": None if not full else np.ctypeslib.as_array(res.pose_flags, (n, P)).copy() if n else np.zeros((0, P), np.uint8),
        "pose_scores": None if not full else np.ctypeslib.as_array(res.pose_scores, (n, P)).copy() if n else np.zeros((0, P), np.float32),
        "n_candidates": nc,
        "n_total_candidates": res.n_total_candidates,
        "ms": (res.ms_candidates, res.ms_images, res.ms_classify),
        "kernel_launches": res.kernel_launches,
    }
    if nc:
        buf = C.string_at(res.candidates, nc * C.sizeof(Pose))
        out["candidates"] = np.frombuffer(buf, dtype=POSE_DTYPE).copy()
    else:
        out["candidates"] = np.zeros(0, dtype=POSE_DTYPE)
    if res.images and nc:
        out["images"] = np.ctypeslib.as_array(res.images, (nc, image_bytes)).copy()
    else:
        out["images"] = None
    return out
