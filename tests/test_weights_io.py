"""Weight import from the reference's other backends' formats (SURVEY.md 8(f).2): `.caffemodel` (Caffe backend) and
OpenVINO IR `.xml` + `.bin` -> the .bin parameter-directory layout (gpdb_read_weights_file / gpdb_load_weights_file).

CPU: the wire-level parsers against files written by this test (a minimal protobuf encoder / an IR skeleton) and against
the reference's own model files, rebuilt byte for byte from tests/golden/ref_model_files.npz, which must reproduce the
shipped .bin parameters bit for bit. GPU: a context loaded from a .caffemodel scores like one given the arrays."""
import os
import struct

import numpy as np
import pytest

from conftest import load_weights
from gpd_b200 import lib
from oracle.reference_data import rebuild_model_file


def _varint(v):
    out = b""
    while True:
        b = v & 0x7F
        v >>= 7
        out += bytes([b | (0x80 if v else 0)])
        if not v:
            return out


def _ld(field, payload):  # length-delimited field
    return _varint((field << 3) | 2) + _varint(len(payload)) + payload


def write_caffemodel(path, blobs, v1=False):
    """caffe.NetParameter with layers conv1, pool1, conv2, ip1, ip2 (LayerParameter: name = 1, type = 2, blobs = 7;
    V1LayerParameter: name = 4, blobs = 6; BlobProto: packed data = 5, shape = 7)."""
    f_layer, f_name, f_blobs = (2, 4, 6) if v1 else (100, 1, 7)
    msg = _ld(1, b"LeNet")
    layers = [("conv1", blobs[0:2]), ("pool1", []), ("conv2", blobs[2:4]), ("ip1", blobs[4:6]), ("ip2", blobs[6:8])]
    for name, bl in layers:
        body = _ld(f_name, name.encode())
        if not v1:
            body += _ld(2, b"Convolution")
        for b in bl:
            shape = _ld(7, _ld(1, b"".join(_varint(int(d)) for d in b.shape)))
            body += _ld(f_blobs, shape + _ld(5, np.ascontiguousarray(b, np.float32).tobytes()))
        msg += _ld(f_layer, body)
    open(path, "wb").write(msg)


def random_net(ch, seed):
    rng = np.random.default_rng(seed)
    f = np.float32
    return [rng.standard_normal((20, ch, 5, 5)).astype(f), rng.standard_normal(20).astype(f),
            rng.standard_normal((50, 20, 5, 5)).astype(f), rng.standard_normal(50).astype(f),
            rng.standard_normal((500, 7200)).astype(f), rng.standard_normal(500).astype(f),
            rng.standard_normal((2, 500)).astype(f), rng.standard_normal(2).astype(f)]


def expected_bin_layout(blobs):
    c1w, c1b, c2w, c2b, f1w, f1b, f2w, f2b = blobs
    ip1 = f1w.reshape(500, 50, 144).transpose(2, 1, 0).reshape(-1)  # [o + 500 (c + 50 j)] = W[o, c 144 + j]
    ip2 = f2w.T.reshape(-1)
    return [c1w.ravel(), c1b, c2w.ravel(), c2b, ip1, f1b, ip2, f2b]


@pytest.mark.parametrize("v1", [False, True])
def test_caffemodel_wire_parser(tmp_path, v1):
    blobs = random_net(3, 1)
    write_caffemodel(tmp_path / "net.caffemodel", blobs, v1=v1)
    arrs, relu = lib.read_weights_file(str(tmp_path / "net.caffemodel"), 3)
    assert relu == -1
    for a, e in zip(arrs, expected_bin_layout(blobs)):
        assert np.array_equal(a, e)
    with pytest.raises(lib.GpdbError) as e:  # wrong channel count is reported, not mis-read
        lib.read_weights_file(str(tmp_path / "net.caffemodel"), 15)
    assert e.value.code == -4 and "expected 7500" in str(e.value)
    open(tmp_path / "junk.caffemodel", "wb").write(b"\xff" * 100)
    with pytest.raises(lib.GpdbError):
        lib.read_weights_file(str(tmp_path / "junk.caffemodel"), 3)
    with pytest.raises(lib.GpdbError):
        lib.read_weights_file(str(tmp_path / "missing.caffemodel"), 3)


def test_openvino_ir_parser(tmp_path):
    blobs = random_net(12, 2)
    raw, xml, off = b"", '<?xml version="1.0" ?>\n<net batch="1" name="model" version="4">\n<layers>\n', 0
    kinds = ["Convolution", "Convolution", "FullyConnected", "FullyConnected"]
    for l in range(4):
        w, b = blobs[2 * l].astype(np.float32).tobytes(), blobs[2 * l + 1].astype(np.float32).tobytes()
        xml += (f'<layer id="{l}" name="{l}" precision="FP32" type="{kinds[l]}"><blobs><weights offset="{off}" size="{len(w)}"/>'
                f'<biases offset="{off + len(w)}" size="{len(b)}"/></blobs></layer>\n')
        if l < 3:
            xml += f'<layer id="{10 + l}" name="r{l}" precision="FP32" type="ReLU"></layer>\n'
        raw += w + b
        off += len(w) + len(b)
    xml += "</layers>\n</net>\n"
    open(tmp_path / "m.xml", "w").write(xml)
    open(tmp_path / "m.bin", "wb").write(raw)
    for wf, mf in ((str(tmp_path / "m.bin"), None), (str(tmp_path / "m.bin"), str(tmp_path / "m.xml")), (str(tmp_path / "m.xml"), None)):
        arrs, relu = lib.read_weights_file(wf, 12, model_file=mf)
        assert relu == 3
        for a, e in zip(arrs, expected_bin_layout(blobs)):
            assert np.array_equal(a, e)


def test_reference_model_files_reproduce_the_bin_parameters(tmp_path, golden_dir):
    """The .caffemodel files of the 15- and 3-channel nets give the reference's .bin parameters (gpd_b200/weights/, equal to
    models/lenet/<ch>channels/params/), the OpenVINO IR of the 12-channel net its ReLU net."""
    g = np.load(os.path.join(golden_dir, "ref_model_files.npz"))
    for ch in (15, 3):
        ref, _ = load_weights(ch)
        arrs, _ = lib.read_weights_file(rebuild_model_file(g, ch, ref, tmp_path), ch)
        assert all(np.array_equal(a, np.ravel(r)) for a, r in zip(arrs, ref)), ch
    w12, _ = load_weights(12)
    arrs, relu = lib.read_weights_file(rebuild_model_file(g, 12, w12, tmp_path), 12)
    assert relu == 3 and all(np.array_equal(a, np.ravel(r)) for a, r in zip(arrs, w12))


@pytest.mark.gpu
def test_context_loaded_from_a_caffemodel_scores_like_the_arrays(tmp_path):
    blobs = random_net(3, 5)
    blobs = [b * s for b, s in zip(blobs, (0.04, 0.1, 0.025, 0.1, 0.008, 0.1, 0.05, 0.1))]
    write_caffemodel(tmp_path / "net.caffemodel", blobs)
    imgs = np.random.default_rng(0).integers(0, 256, (64, 60, 60, 3), dtype=np.uint8)
    a = lib.Context(lib.default_params(channels=3))
    a.load_weights_file(str(tmp_path / "net.caffemodel"))
    b = lib.Context(lib.default_params(channels=3))
    b.set_weights(expected_bin_layout(blobs))
    sa, la = a.classify(imgs)
    sb, lb = b.classify(imgs)
    assert np.array_equal(la, lb) and np.array_equal(sa, sb)
    with pytest.raises(lib.GpdbError):
        a.load_weights_file(str(tmp_path / "nope.weights"))
    a.close()
    b.close()
