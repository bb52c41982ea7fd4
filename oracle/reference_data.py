"""Helpers shared by the tests and tools/make_goldens.py for the data stored from the original GPD project under
tests/golden: the cases of the cfg-parser comparison and the rebuilding of the reference's model files.

TEST INFRASTRUCTURE ONLY, like the rest of oracle/: nothing under gpd_b200/ imports it."""
import ctypes as C
import hashlib
import os

import numpy as np

TRICKY_CFG = ("# comment line\n\n   \nalpha = 1.5\nbeta=2\n\tgamma\t=\t3.25   # trailing comment\n  delta   =  a b  c  \nalpha = 99\n"
              "vec = 0.1 -2 3e-3 4\nflag0 = 0\nflag1 = 1\nempty_after_hash = #nothing\nint_as_float = 7.9\nweights_file = ../x/y/\n"
              "spaced key = 5\n")
TRICKY_KEYS = ("alpha", "beta", "gamma", "delta", "vec", "flag0", "flag1", "empty_after_hash", "int_as_float", "weights_file", "spaced",
               "spaced key", "missing")
SHIPPED_CFGS = ("eigen_params.cfg", "caffe_params.cfg", "vino_params_12channels.cfg", "hand_geometry.cfg", "image_geometry_15channels.cfg",
                "ros_eigen_params.cfg")
SHIPPED_KEYS = ("hand_geometry_filename", "image_geometry_filename", "weights_file", "model_file", "workspace", "workspace_grasps",
                "num_samples", "num_threads", "voxelize", "voxel_size", "hand_axes", "finger_width", "hand_outer_diameter",
                "volume_width", "image_num_channels", "camera_position", "min_inliers", "num_selected", "direction", "thresh_rad")
GEOMETRY_CFGS = ("hand_geometry.cfg", "ur5_hand_geometry.cfg", "image_geometry_15channels.cfg", "image_geometry_12channels.cfg",
                 "image_geometry_3channels.cfg", "image_geometry_1channels.cfg", "eigen_params.cfg")


def config_parser_answers(L, ref, cfg_dir, tmp_dir):
    """Every value a util::ConfigFile / candidate::HandGeometry / descriptor::ImageGeometry implementation returns on a cfg
    with the format's corner cases, a missing file and the shipped cfg files in `cfg_dir`, keyed "<file>|<key>".
    L is the shim's libgpd_host.so, or with ref = True the reference's own parser (oracle/_ref/libgpd_ref_config.so,
    whose answers tools/make_goldens.py stores in tests/golden/ref_config_parser.json)."""
    pre, suf = ("gpdref_config_get", ("_double", "_int", "_bool", "_doubles")) if ref else ("gpdConfigGet", ("Double", "Int", "Bool", "Doubles"))
    getattr(L, pre).argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int]
    for s, t in zip(suf[:3], (C.c_double, C.c_int, C.c_int)):
        f = getattr(L, pre + s)
        f.argtypes, f.restype = [C.c_char_p, C.c_char_p, t], t
    getattr(L, pre + suf[3]).argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_int]

    def get(path, key):
        p, k = path.encode(), key.encode()
        buf = C.create_string_buffer(512)
        found = getattr(L, pre)(p, k, b"<default>", buf, 512)
        vec = (C.c_double * 16)()
        nv = getattr(L, pre + suf[3])(p, k, b"1.5 2.5", vec, 16)
        return [found, buf.value.decode(), getattr(L, pre + suf[0])(p, k, -7.25), getattr(L, pre + suf[1])(p, k, -7),
                getattr(L, pre + suf[2])(p, k, 1), nv, list(vec[:min(nv, 16)])]
    tricky, missing = os.path.join(tmp_dir, "tricky.cfg"), os.path.join(tmp_dir, "does_not_exist.cfg")
    with open(tricky, "w") as f:
        f.write(TRICKY_CFG)
    out = {f"tricky.cfg|{k}": get(tricky, k) for k in TRICKY_KEYS}
    for name in SHIPPED_CFGS:
        out.update({f"{name}|{k}": get(os.path.join(cfg_dir, name), k) for k in SHIPPED_KEYS})
    out["does_not_exist.cfg|alpha"] = get(missing, "alpha")
    hg, ig = ("gpdref_hand_geometry", "gpdref_image_geometry") if ref else ("gpdHandGeometry", "gpdImageGeometry")
    for path in [tricky, missing] + [os.path.join(cfg_dir, n) for n in GEOMETRY_CFGS]:
        a, b, c2 = (C.c_double * 5)(), (C.c_double * 3)(), (C.c_int * 2)()
        getattr(L, hg)(path.encode(), a)
        getattr(L, ig)(path.encode(), b, c2)
        out[os.path.basename(path) + "|geometry"] = [list(a), list(b), list(c2)]
    return out


# the reference's model files of the three shipped nets (models/caffe/<ch>channels/, models/openvino/), by channel count
MODEL_FILES = {15: "two_views_15_channels_90_deg_no_flipping.caffemodel", 3: "bottles_boxes_cans_5xNeg.caffemodel",
               12: "two_views_12_channels_curv_axis.bin"}


def blob_layout(arrays):
    """Inverse of tests/test_weights_io.py:expected_bin_layout: the eight .bin-layout arrays as the flat blobs of a .caffemodel / an IR .bin."""
    c1w, c1b, c2w, c2b, ip1, f1b, ip2, f2b = [np.ravel(a).astype(np.float32) for a in arrays]
    return [c1w, c1b, c2w, c2b, ip1.reshape(144, 50, 500).transpose(2, 1, 0).reshape(-1), f1b, ip2.reshape(500, 2).T.reshape(-1), f2b]


def rebuild_model_file(golden, ch, arrays, d):
    """Writes the reference's model file of the `ch`-channel net into directory d: its skeleton (the file without the eight
    weight payloads) with the payloads of `arrays` put back at the stored offsets, plus the IR's .xml. The result must hash
    to the stored SHA-256 of the reference's file."""
    skel, blobs = golden[f"{ch}_skeleton"].tobytes(), blob_layout(arrays)
    out, s, end = bytearray(), 0, 0
    for off, k, nbytes in golden[f"{ch}_cuts"]:
        out += skel[s:s + off - end]
        s += off - end
        assert blobs[k].nbytes == nbytes
        out += blobs[k].tobytes()
        end = off + nbytes
    out += skel[s:]
    assert hashlib.sha256(out).hexdigest() == str(golden[f"{ch}_sha256"]), MODEL_FILES[ch]
    path = os.path.join(d, MODEL_FILES[ch])
    open(path, "wb").write(out)
    if f"{ch}_xml" in golden:
        open(os.path.splitext(path)[0] + ".xml", "wb").write(golden[f"{ch}_xml"].tobytes())
    return path
