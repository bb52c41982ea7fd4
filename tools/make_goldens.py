#!/usr/bin/env python
"""Generate the committed fixtures under tests/golden/ and gpd_b200/weights/.

Runs ONLY in the build container (it reads /root/reference and uses cv2 / cv2.dnn as the
independent ground truth the reference itself links against). The GPU box never runs this.

  tests/golden/krylon_voxel.npz      tutorials/krylon.pcd voxelised + normals (input fixture)
  tests/golden/cv_pins.npz           cv2.dilate / cv2.normalize / convertTo(CV_8U) known answers
  tests/golden/lenet_caffe_{15,3}ch.npz   cv2.dnn forward of the reference .prototxt/.caffemodel
  tests/golden/lenet_ir_12ch.npz     torch restatement of the OpenVINO IR 12-channel net
  tests/golden/krylon_oracle_15ch.npz     oracle outputs (regression pin of the oracle itself)
  gpd_b200/weights/lenet_{15,3,12}ch.npz  the reference weights in the .bin layout
  tests/golden/krylon_preprocess.npz      raw tutorials/krylon.pcd points + the oracle's preprocessing outputs
                                          + an independent float64 PCA normal per point (`--only preprocess`)
  tests/golden/cfg/*.cfg                  the reference's cfg files the parser tests read, and
  tests/golden/ref_config_parser.json     what the reference's own cfg parser (oracle/_ref) answers on them (`--only ref_config`)
  tests/golden/ref_model_files.npz        the reference's .caffemodel / IR files of the shipped nets without their weight
                                          payloads, which tests rebuild from gpd_b200/weights/ (`--only ref_models`)
"""
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gpd_b200 import abi, scenes  # noqa: E402
from oracle import oracle  # noqa: E402

REF = "/root/reference"
G = os.path.join(ROOT, "tests", "golden")
W = os.path.join(ROOT, "gpd_b200", "weights")
NAMES = oracle.WeightPack.NAMES


def save_weights(ch, arrays, relu_after_conv):
    np.savez(os.path.join(W, f"lenet_{ch}ch.npz"), relu_after_conv=np.int32(relu_after_conv),
             **{n: a for n, a in zip(NAMES, arrays)})


def caffe_net(ch):
    import cv2
    d = f"{REF}/models/caffe/{ch}channels/"
    proto = open(d + f"lenet_{ch}_channels.prototxt").read()
    proto = re.sub(r"^input:.*$", "", proto, flags=re.M)
    i = proto.index("layer")
    j = proto.index("layer", i + 5)
    proto = proto[:i] + f'input: "data"\ninput_shape {{ dim: 1 dim: {ch} dim: 60 dim: 60 }}\n' + proto[j:]
    f = tempfile.NamedTemporaryFile("w", suffix=".prototxt", delete=False)
    f.write(proto)
    f.close()
    model = d + ("two_views_15_channels_90_deg_no_flipping.caffemodel" if ch == 15 else "bottles_boxes_cans_5xNeg.caffemodel")
    return cv2.dnn.readNetFromCaffe(f.name, model)


def test_images(ch, n, seed):
    rng = np.random.default_rng(seed)
    imgs = rng.integers(0, 256, (n, 60, 60, ch), dtype=np.uint8)
    half = n // 2
    imgs[:half] = ((rng.random((half, 60, 60, ch)) < 0.3) * imgs[:half]).astype(np.uint8)
    return imgs


def lenet_caffe(ch):
    net = caffe_net(ch)
    arrays = scenes.load_weights_dir(f"{REF}/models/lenet/{ch}channels/params/")
    save_weights(ch, arrays, 0)
    imgs = test_images(ch, 12, ch)
    out = []
    for b in imgs.transpose(0, 3, 1, 2).astype(np.float32):
        net.setInput(b[None])
        out.append(net.forward().ravel().copy())
    out = np.array(out, np.float32)
    p = abi.default_params(ch)
    sc, lg = oracle.classify(p, oracle.WeightPack(arrays), imgs)
    rel = np.abs(out - lg).max() / np.abs(out).max()
    print(f"lenet {ch}ch: oracle vs cv2.dnn caffe max rel diff {rel:.3e}")
    assert rel < 1e-5
    np.savez_compressed(os.path.join(G, f"lenet_caffe_{ch}ch.npz"), images=imgs, logits=out)


def lenet_ir_12ch():
    """models/openvino/two_views_12_channels_curv_axis.{xml,bin}: conv1(12->20,k5)+ReLU+pool,
    conv2(20->50)+ReLU+pool, FC 500+ReLU, FC 2 (pytorch/network.py:32-47). Blob offsets from the
    XML. Converted into the Eigen .bin layout (ip weights column-major (out,in), ip1 input index
    k = c + 50*j) so the library needs only relu_after_conv=1."""
    import torch
    import torch.nn.functional as F
    xml = open(f"{REF}/models/openvino/two_views_12_channels_curv_axis.xml").read()
    offs = [(int(a), int(b)) for a, b in re.findall(r'<(?:weights|biases) offset="(\d+)" size="(\d+)"', xml)]
    raw = open(f"{REF}/models/openvino/two_views_12_channels_curv_axis.bin", "rb").read()
    blobs = [np.frombuffer(raw[o:o + s], dtype=np.float32).copy() for o, s in offs]
    sizes = [len(b) for b in blobs]
    print("IR blobs", offs, sizes)
    c1w, c1b, c2w, c2b, f1w, f1b, f2w, f2b = blobs
    assert sizes == [20 * 12 * 25, 20, 50 * 20 * 25, 50, 500 * 7200, 500, 1000, 2], sizes
    # torch reference forward (CHW flatten, row-major (out,in) FC weights)
    imgs = test_images(12, 12, 12)
    x = torch.from_numpy(imgs.transpose(0, 3, 1, 2).astype(np.float32)).double()
    t = lambda a, s: torch.from_numpy(a.reshape(s)).double()  # noqa: E731
    h = F.max_pool2d(F.relu(F.conv2d(x, t(c1w, (20, 12, 5, 5)), t(c1b, (20,)))), 2)
    h = F.max_pool2d(F.relu(F.conv2d(h, t(c2w, (50, 20, 5, 5)), t(c2b, (50,)))), 2)
    h = F.relu(F.linear(h.reshape(len(imgs), -1), t(f1w, (500, 7200)), t(f1b, (500,))))
    y = F.linear(h, t(f2w, (2, 500)), t(f2b, (2,))).float().numpy()
    # -> .bin layout: ip1[o + 500*(c + 50*j)] = f1w[o, c*144 + j]; ip2[o + 2*k] = f2w[o, k]
    ip1 = f1w.reshape(500, 50, 144).transpose(2, 1, 0).reshape(-1).copy()
    ip2 = f2w.reshape(2, 500).T.reshape(-1).copy()
    arrays = [c1w, c1b, c2w, c2b, ip1, f1b, ip2, f2b]
    save_weights(12, arrays, 1)
    p = abi.default_params(12, relu_after_conv=1)
    sc, lg = oracle.classify(p, oracle.WeightPack(arrays), imgs)
    rel = np.abs(y - lg).max() / np.abs(y).max()
    print(f"lenet 12ch IR: oracle vs torch float64 max rel diff {rel:.3e}")
    assert rel < 1e-5
    np.savez_compressed(os.path.join(G, "lenet_ir_12ch.npz"), images=imgs, logits=y)


def cv_pins():
    import cv2
    rng = np.random.default_rng(0)
    ins, outs = [], []
    el = cv2.getStructuringElement(cv2.MORPH_RECT, (3, 3))
    for trial in range(24):
        ch = 3 if trial % 2 else 1
        img = np.zeros((60, 60, ch), np.float32)
        m = rng.random((60, 60)) < rng.uniform(0.02, 0.9)
        vals = rng.random((60, 60, ch)).astype(np.float32)
        if trial % 5 == 0:
            vals += 0.3
        if trial % 7 == 0:
            m[:] = True
        if trial == 23:
            m[:] = False
        img[m] = vals[m]
        d = cv2.dilate(img, el).reshape(60, 60, ch)
        nrm = cv2.normalize(d, None, 0.0, 1.0, cv2.NORM_MINMAX, cv2.CV_32F).reshape(60, 60, ch)
        u8 = cv2.convertScaleAbs(nrm, alpha=255.0).reshape(60, 60, ch)
        pad = np.zeros((60, 60, 3), np.float32)
        pad[:, :, :ch] = img
        padu = np.zeros((60, 60, 3), np.uint8)
        padu[:, :, :ch] = u8
        ins.append(pad)
        outs.append(padu)
    np.savez_compressed(os.path.join(G, "cv_pins.npz"), inputs=np.array(ins), outputs=np.array(outs),
                        channels=np.array([3 if t % 2 else 1 for t in range(24)], np.int32))


def krylon_oracle():
    k = scenes.krylon_cloud(f"{REF}/tutorials/krylon.pcd")
    np.savez_compressed(os.path.join(G, "krylon_voxel.npz"), **k)
    oc = oracle.OracleCloud(k["xyz"], k["normals"], k["cam_source"], k["view_points"])
    arrays = scenes.load_weights_dir(f"{REF}/models/lenet/15channels/params/")
    p = abi.default_params(15, keep_images=1)
    sidx = scenes.sample_indices(2, len(k["xyz"]), 24)
    r = oc.detect(p, oracle.WeightPack(arrays), sidx)
    crc = np.array([zlib.crc32(im.tobytes()) for im in r["images"]], np.uint32)
    np.savez_compressed(os.path.join(G, "krylon_oracle_15ch.npz"), sample_idx=sidx, frames=r["frames"],
                        frame_valid=r["frame_valid"], pose_flags=r["pose_flags"], pose_scores=r["pose_scores"],
                        candidates=r["candidates"], image_crc32=crc, images_first4=r["images"][:4])
    print("krylon oracle golden:", r["n_candidates"], "candidates")


def krylon_preprocess():
    """Raw tutorial cloud -> CandidatesGenerator::preprocessPointCloud (oracle restatement) with the defaults of
    cfg/eigen_params.cfg:16-21; `pca64` = normal direction from numpy float64 eigh of the same r-ball (independent
    of the float32 PCL restatement; agreement is limited by PCL's float32 single-pass covariance, ~1e-4)."""
    from scipy.spatial import cKDTree
    raw = scenes.load_pcd_ascii(f"{REF}/tutorials/krylon.pcd")
    vp = np.zeros((1, 3))
    pp = abi.default_preprocess_params()
    r = oracle.preprocess(raw, None, vp, pp)
    P = r["xyz"].astype(np.float64)
    tree = cKDTree(P)
    pca = np.zeros_like(P)
    for i in range(len(P)):
        d2 = ((P - P[i]) ** 2).sum(1)
        nb = np.nonzero(d2 < 0.03 ** 2)[0]
        w, v = np.linalg.eigh(np.cov(P[nb].T, bias=True))
        pca[i] = v[:, 0]
    np.savez_compressed(os.path.join(G, "krylon_preprocess.npz"), raw=raw, xyz=r["xyz"], normals=r["normals"],
                        cam_source=r["cam_source"], src=r["src"], pca64=pca)
    print("krylon_preprocess:", len(raw), "->", len(P))


def ref_config():
    """The cfg files of the parser tests (oracle/reference_data.py), and the answers of the reference's own util::ConfigFile /
    HandGeometry / ImageGeometry (oracle/_ref, built from the reference's sources) on them."""
    import ctypes
    from oracle import reference_data as t
    cfg = os.path.join(G, "cfg")
    os.makedirs(cfg, exist_ok=True)
    for name in sorted(set(t.SHIPPED_CFGS + t.GEOMETRY_CFGS + ("vino_params_12channels.cfg", "all_axes_vino_12channels.cfg",
                                                                "image_geometry_12channels.cfg"))):
        shutil.copyfile(f"{REF}/cfg/{name}", os.path.join(cfg, name))
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "_ref", f"REF={REF}", "-s"])
    R = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libgpd_ref_config.so"))
    with tempfile.TemporaryDirectory() as d:
        ans = t.config_parser_answers(R, True, cfg, d)
    with open(os.path.join(G, "ref_config_parser.json"), "w") as f:
        json.dump(ans, f, indent=0, sort_keys=True)
    print("ref_config_parser:", len(ans), "answers")


def ref_models():
    """Each model file of oracle/reference_data.MODEL_FILES as a skeleton (the file with its eight weight payloads cut out), the
    payloads' offsets, the file's SHA-256 and, for the IR, its .xml. The payloads are the committed weights in the blob
    layout, which this checks against the reference's .bin parameters."""
    from oracle.reference_data import MODEL_FILES, blob_layout
    out = {}
    for ch, name in MODEL_FILES.items():
        ir = name.endswith(".bin")
        raw = open(f"{REF}/models/{'openvino' if ir else f'caffe/{ch}channels'}/{name}", "rb").read()
        z = np.load(os.path.join(W, f"lenet_{ch}ch.npz"))
        w = [z[n] for n in NAMES]
        if not ir:
            ref = scenes.load_weights_dir(f"{REF}/models/lenet/{ch}channels/params/")
            assert all(np.array_equal(np.ravel(a), r) for a, r in zip(w, ref)), ch
        skel, cuts, pos = bytearray(), [], 0
        for k, b in enumerate(blob_layout(w)):
            off = raw.find(b.tobytes(), pos)
            assert off >= 0, (name, NAMES[k])
            skel += raw[pos:off]
            cuts.append((off, k, b.nbytes))
            pos = off + b.nbytes
        skel += raw[pos:]
        out[f"{ch}_skeleton"] = np.frombuffer(bytes(skel), np.uint8)
        out[f"{ch}_cuts"] = np.array(cuts, np.int64)
        out[f"{ch}_sha256"] = np.array(hashlib.sha256(raw).hexdigest())
        if ir:
            out[f"{ch}_xml"] = np.frombuffer(open(f"{REF}/models/openvino/{name[:-4]}.xml", "rb").read(), np.uint8)
        print(f"{name}: {len(raw)} bytes -> {len(skel)} byte skeleton")
    np.savez_compressed(os.path.join(G, "ref_model_files.npz"), **out)


if __name__ == "__main__":
    os.makedirs(G, exist_ok=True)
    os.makedirs(W, exist_ok=True)
    only = {"preprocess": krylon_preprocess, "ref_config": ref_config, "ref_models": ref_models}
    if "--only" in sys.argv:
        only[sys.argv[sys.argv.index("--only") + 1]]()
        sys.exit(0)
    krylon_oracle()
    cv_pins()
    lenet_caffe(15)
    lenet_caffe(3)
    lenet_ir_12ch()
    ref_config()
    ref_models()
