"""Host-side logic of the drop-in boundary, runnable without a GPU: the text-format reader, the
Caffe-API mirror's Net construction (split insertion, blob names and shapes, output order,
parameter shapes), the generated model zoo, and the exported C ABI."""
import hashlib
import json
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle.build_ref import REF, present

ROOT = Path(__file__).resolve().parent.parent
REF_EX = REF / "examples"
GOLD = Path(__file__).resolve().parent / "golden"


def test_capi_exports_every_declared_symbol():
    from mscnn_b200 import capi
    L = capi.lib()
    hdr = (ROOT / "include" / "mscnn_b200.h").read_text()
    names = sorted(set(re.findall(r"\b(mscnn_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, f"declared in include/mscnn_b200.h but not exported: {missing}"
    assert b"sm_100a" in L.mscnn_version()


def test_library_carries_sm100a_tensor_core_code():
    out = subprocess.run(["cuobjdump", "-sass", str(ROOT / "mscnn_b200" / "libmscnn_b200.so")],
                         capture_output=True, text=True).stdout
    if not out:
        pytest.skip("cuobjdump unavailable")
    assert "UTCHMMA" in out and "UTMALDG" in out and "UTMASTG" in out and "LDTM" in out


def test_only_the_pair_kernel_contains_cluster_instructions():
    """A kernel that contains cta_group::2 / cluster instructions can only be launched as a cluster ("cluster
    misconfiguration" otherwise): the CTA-pair build of the convolution kernel must be its own instantiation, and it
    must really carry the 2-CTA tensor-core instructions."""
    out = subprocess.run(["cuobjdump", "-sass", str(ROOT / "mscnn_b200" / "libmscnn_b200.so")],
                         capture_output=True, text=True).stdout
    if not out:
        pytest.skip("cuobjdump unavailable")
    users, fn = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
        elif fn and re.search(r"\b(UTCHMMA\.2CTA|UTCATOMSWS\.2CTA|UCGABAR_ARV|UCGABAR_WAIT)", line):
            users[fn] = users.get(fn, 0) + 1
    assert users, "no 2-CTA instructions in the library: the CTA-pair kernel is missing"
    assert all("conv_igemm_kernelILi256ELb1" in f for f in users), sorted(users)
    assert any("UTCHMMA.2CTA" in l for l in out.splitlines())


def test_net_kitti_8s_structure():
    from mscnn_b200 import models
    from mscnn_b200.net import Net
    net = Net(models.kitti(768, 2560, 8))
    assert net.inputs == ["data"]
    assert net.outputs == ["bbox_pred", "cls_pred", "proposals_score"]       # name order, net.cpp:268-274
    # InsertSplits names after the LAST writer (the in-place ReLU), insert_splits.cpp:37-40,110-124
    for k in range(4):
        assert f"conv4_3_relu4_3_0_split_{k}" in net.blob_names
    assert "proposals_proposals_0_split_0" in net.blob_names
    assert net.blob_shape("data") == (1, 3, 768, 2560)
    assert net.blob_shape("conv1_2") == (1, 64, 768, 2560)
    assert net.blob_shape("conv4_3") == (1, 512, 96, 320)
    assert net.blob_shape("pool6") == (1, 512, 12, 40)
    assert net.blob_shape("LFCN_4_7x7") == (1, 9, 12, 40)
    assert net.blob_shape("proposals") == (1, 5, 1, 1)                       # dummy reshape
    assert net.blob_shape("roi_pool") == (1, 1024, 7, 7)
    assert net.blob_shape("roi_c1") == (1, 512, 5, 5)
    assert net.blob_shape("fc6") == (1, 4096) and net.blob_shape("bbox_pred") == (1, 20)
    assert net.param_shapes("conv1_1") == [(64, 3, 3, 3), (64,)]
    assert net.param_shapes("LFCN_1_7x7") == [(9, 512, 7, 7), (9,)]
    assert net.param_shapes("fc6") == [(4096, 12800), (4096,)]
    assert net.layer_types.count("Split") == 7   # conv4_3, loss1_conv1, conv5_3, conv6_1, pool6, proposals, fc6


def test_net_reshape_input_propagates():
    from mscnn_b200 import models
    from mscnn_b200.net import Net
    net = Net(models.kitti(576, 1920, 7, up2x=True))
    net.reshape_input("data", 2, 3, 192, 640)
    assert net.blob_shape("conv4_3") == (2, 512, 24, 80)
    assert net.blob_shape("conv4_3_2x") == (2, 512, 48, 160)
    assert net.blob_shape("LFCN_4_5x5") == (2, 9, 3, 10)


def test_widerface_structure():
    from mscnn_b200 import models
    from mscnn_b200.net import Net
    net = Net(models.widerface(768, 1024, batch=2))
    assert net.blob_shape("LFCN_1_12x12") == (2, 6, 96, 128)
    assert net.blob_shape("pool6") == (2, 512, 12, 16)
    assert net.blob_shape("roi_c1") == (1, 512, 5, 5) and net.blob_shape("fc6") == (1, 2048)
    assert net.param_shapes("conv4_3_2x") == [(512, 1, 4, 4)]


def test_prototxt_syntax_quirks():
    """Comments (also trailing), `field: { }` and `field { }`, several pairs per line, negative and
    float values, enums and strings -- all present in the shipped deploy files (SURVEY.md section 7)."""
    from mscnn_b200.net import Net
    text = '''name: "q"  # a comment
input: "data" input_dim: 1 input_dim: 64 input_dim: 8 input_dim: 8
layer { bottom: "data" top: "c" name: "c" type: "Convolution"
  param { lr_mult: 1 decay_mult: 1 } param { lr_mult: 2 decay_mult: 0 }
  convolution_param { num_output: 6 kernel_size: 3
    #pad: 1
    weight_filler: { type: "gaussian" std: 0.01 } bias_filler { type: "constant" value: -0.5 } } }
layer { bottom: "c" top: "p" name: "p" type: "Pooling" pooling_param { pool: AVE kernel_size: 2 stride: 2 } propagate_down: 0 }
'''
    net = Net(text)
    assert net.blob_shape("c") == (1, 6, 6, 6) and net.blob_shape("p") == (1, 6, 3, 3)


def test_unknown_field_is_rejected():
    from mscnn_b200 import capi
    from mscnn_b200.net import Net
    with pytest.raises(capi.MscnnError):
        Net('input: "d" input_dim: 1 input_dim: 1 input_dim: 4 input_dim: 4\n'
            'layer { bottom: "d" top: "p" name: "p" type: "Pooling" pooling_param { kernel_size: 2 bogus_field: 3 } }\n')


SHIPPED_DEPLOY = [
    ("kitti_car/mscnn-8s-768-trainval", ("kitti", (768, 2560, 8, False))),
    ("kitti_car/mscnn-7s-576", ("kitti", (576, 1920, 7, False))),
    ("kitti_car/mscnn-7s-576-2x", ("kitti", (576, 1920, 7, True))),
    ("widerface/mscnn-12s-2x", ("widerface", (512, 512))),
    ("kitti_car/cascade-mscnn-7s-576-2x", ("kitti_cascade", (576, 1920))),
    ("widerface/cascade-mscnn-12s-align", ("widerface_cascade", (512, 512))),
]


def net_structure(net):
    """sha256 of the canonical JSON of each thing a loaded net exposes: wiring, parameter and blob shapes, the settings
    of every layer."""
    parts = {"layer_names": net.layer_names, "layer_types": net.layer_types, "blob_names": net.blob_names,
             "layers": net.layers(), "blob_shapes": [net.blob_shape(b) for b in net.blob_names],
             "layer_param_strings": net.layer_param_strings()}
    return {k: hashlib.sha256(json.dumps(v).encode()).hexdigest() for k, v in parts.items()}


@pytest.mark.parametrize("ref_path,gen", SHIPPED_DEPLOY)
def test_shipped_deploy_files_load_unchanged_and_match_generated(ref_path, gen):
    """The reference's shipped <ref_path>/mscnn_deploy.prototxt, loaded unchanged, is recorded in
    tests/golden/shipped_deploy_nets.json (tests/golden/make_golden.py deploy); the generated net must equal it."""
    from mscnn_b200 import models
    from mscnn_b200.net import Net
    shipped = json.loads((GOLD / "shipped_deploy_nets.json").read_text())[ref_path]
    generated = net_structure(Net(getattr(models, gen[0])(*gen[1])))
    for part, digest in shipped.items():
        assert generated[part] == digest, part


@pytest.mark.skipif(not present(REF_EX), reason="the reference tree is not readable here")
def test_every_shipped_deploy_net_loads():
    """All 23 mscnn_deploy.prototxt files of the reference's model zoo (KITTI car / ped-cyc, Caltech,
    CityPersons, WIDER FACE, plain and cascade) parse, wire up and shape-infer unchanged."""
    from mscnn_b200.net import Net
    files = sorted(REF_EX.glob("*/*/mscnn_deploy.prototxt"))
    assert len(files) == 23
    for f in files:
        net = Net(str(f))
        assert net.blob_shape("proposals") == (1, 5, 1, 1)      # BoxOutput's dummy reshape
        assert "data" in net.blob_names


def test_fused_groups_are_static():
    """The fusion pass records who does a folded layer's work: pool1/2/3 -> their convolution, the context ROIPooling ->
    the object one (the group's leader); everything else does its own.  ForwardFromTo widens a range start to it."""
    from mscnn_b200 import models
    from mscnn_b200.net import Net
    net = Net(models.kitti(96, 320, 8, False, batch=1))
    assert net.fused_producer("pool1") == "conv1_2" and net.fused_producer("pool2") == "conv2_2"
    assert net.fused_producer("pool3") == "conv3_3"
    assert net.fused_producer("pool4") == "pool4"            # reads conv4_3 through a Split top: not folded
    assert net.fused_producer("roi_pool_ctx") == "roi_pool_org" and net.fused_producer("roi_pool_org") == "roi_pool_org"
    assert net.fused_producer("conv4_3") == "conv4_3" and net.fused_producer("fc6") == "fc6"


def test_params_shared_by_name():
    """ParamSpec names make layers share one blob (Net::AppendParam, net.cpp:448-538): the cascade
    nets' third-stage ensemble heads reuse the first- and second-stage weights."""
    from mscnn_b200 import models
    from mscnn_b200.net import Net
    net = Net(models.widerface_cascade(128, 192))
    w = np.full(net.param_shapes("cls_pred")[0], 0.25, dtype=np.float32)
    net.set_params({"cls_pred": [w, np.arange(2, dtype=np.float32)]})
    assert np.array_equal(net.param("cls_pred_1st_3rd", 0), w)
    assert np.array_equal(net.param("cls_pred_1st_3rd", 1), [0, 1])
    assert not np.array_equal(net.param("cls_pred_2nd_3rd", 0), w)       # shares with cls_pred_2nd instead
    net.set_params({"cls_pred_2nd_3rd": [2 * w, np.zeros(2, dtype=np.float32)]})
    assert np.array_equal(net.param("cls_pred_2nd", 0), 2 * w)
    # a shape mismatch between sharers is a CHECK failure (net.cpp:497-509): it aborts like Caffe does
    bad = ('input: "d" input_dim: 1 input_dim: 4 input_dim: 1 input_dim: 1\n'
           'layer { name: "a" type: "InnerProduct" bottom: "d" top: "a" param { name: "w" } inner_product_param { num_output: 3 } }\n'
           'layer { name: "b" type: "InnerProduct" bottom: "d" top: "b" param { name: "w" } inner_product_param { num_output: 2 } }\n')
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", "import sys; from mscnn_b200.net import Net; Net(sys.argv[1])", bad],
                       capture_output=True, text=True, cwd=str(Path(__file__).resolve().parents[1]))
    assert r.returncode != 0 and "Cannot share param" in r.stderr


def test_synth_is_deterministic_and_name_keyed():
    from mscnn_b200 import synth
    layers = [("conv1_1", "Convolution", [(64, 3, 3, 3), (64,)]), ("LFCN_1_5x5", "Convolution", [(9, 512, 5, 5), (9,)]),
              ("conv4_3_2x", "Deconvolution", [(512, 1, 4, 4)])]
    a, b = synth.make_weights(layers), synth.make_weights(list(reversed(layers)))
    for k in a:
        assert all(np.array_equal(x, y) for x, y in zip(a[k], b[k]))
    assert a["LFCN_1_5x5"][1][0] == synth.BG_BIAS and a["conv4_3_2x"][0][5, 0, 1, 1] == np.float32(0.5625)
    img = synth.make_images(2, 8, 8)
    assert img.shape == (2, 3, 8, 8) and img[0, 0].max() <= 255 - 104 and img[0, 2].min() >= -123
    assert np.array_equal(synth.make_images(1, 8, 8, first_index=1)[0], img[1])


# ---- .caffemodel (NetParameter wire format) reader: Net::CopyTrainedLayersFrom, net.cpp:787-803 ----
def _varint(v: int) -> bytes:
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _ld(field: int, payload: bytes) -> bytes:
    return _varint((field << 3) | 2) + _varint(len(payload)) + payload


def _blob_proto(arr: np.ndarray, legacy: bool = False) -> bytes:
    a = np.ascontiguousarray(arr, dtype="<f4")
    if legacy:   # num/channels/height/width fields 1..4 (old caffemodels)
        dims = list(a.shape) + [1] * (4 - a.ndim)
        msg = b"".join(_varint((i + 1) << 3) + _varint(d) for i, d in enumerate(dims))
    else:        # BlobShape shape = 7 { repeated int64 dim = 1 [packed] }
        msg = _ld(7, _ld(1, b"".join(_varint(d) for d in a.shape)))
    return msg + _ld(5, a.tobytes())


def _caffemodel(layers: dict, legacy=False) -> bytes:
    out = _ld(1, b"net")
    for name, blobs in layers.items():
        lp = _ld(1, name.encode()) + _ld(2, b"Convolution") + b"".join(_ld(7, _blob_proto(b, legacy)) for b in blobs)
        out += _ld(100, lp)
    return out


def _caffe_pb():
    """NetParameter / LayerParameter / V1LayerParameter / BlobProto / BlobShape message classes built with the
    google.protobuf RUNTIME from a descriptor written out by hand from the reference's schema (no protoc in the image):
    /root/reference/src/caffe/proto/caffe.proto:5-24 (BlobShape, BlobProto), :64-100 (NetParameter: name = 1,
    layers = 2, layer = 100), :310-330 (LayerParameter: name = 1, type = 2, bottom = 3, top = 4, blobs = 7),
    V1LayerParameter (bottom = 2, top = 3, name = 4, type = 5 (enum), blobs = 6).  An encoder independent of the
    library's own reader and of the hand encoder above."""
    from google.protobuf import descriptor_pb2, descriptor_pool, message_factory
    F = descriptor_pb2.FieldDescriptorProto
    fd = descriptor_pb2.FileDescriptorProto(name="caffe_subset.proto", package="caffe_subset", syntax="proto2")

    def msg(name, fields):
        m = fd.message_type.add(name=name)
        for fname, num, ftype, label, extra in fields:
            f = m.field.add(name=fname, number=num, type=ftype, label=label)
            if extra.get("packed"):
                f.options.packed = True
            if "type_name" in extra:
                f.type_name = ".caffe_subset." + extra["type_name"]
    O, R = F.LABEL_OPTIONAL, F.LABEL_REPEATED
    msg("BlobShape", [("dim", 1, F.TYPE_INT64, R, {"packed": True})])
    msg("BlobProto", [("shape", 7, F.TYPE_MESSAGE, O, {"type_name": "BlobShape"}),
                      ("data", 5, F.TYPE_FLOAT, R, {"packed": True}), ("diff", 6, F.TYPE_FLOAT, R, {"packed": True}),
                      ("double_data", 8, F.TYPE_DOUBLE, R, {"packed": True}),
                      ("num", 1, F.TYPE_INT32, O, {}), ("channels", 2, F.TYPE_INT32, O, {}),
                      ("height", 3, F.TYPE_INT32, O, {}), ("width", 4, F.TYPE_INT32, O, {})])
    msg("LayerParameter", [("name", 1, F.TYPE_STRING, O, {}), ("type", 2, F.TYPE_STRING, O, {}),
                           ("bottom", 3, F.TYPE_STRING, R, {}), ("top", 4, F.TYPE_STRING, R, {}),
                           ("blobs", 7, F.TYPE_MESSAGE, R, {"type_name": "BlobProto"})])
    msg("V1LayerParameter", [("bottom", 2, F.TYPE_STRING, R, {}), ("top", 3, F.TYPE_STRING, R, {}),
                             ("name", 4, F.TYPE_STRING, O, {}), ("type", 5, F.TYPE_INT32, O, {}),
                             ("blobs", 6, F.TYPE_MESSAGE, R, {"type_name": "BlobProto"})])
    msg("NetParameter", [("name", 1, F.TYPE_STRING, O, {}),
                         ("layers", 2, F.TYPE_MESSAGE, R, {"type_name": "V1LayerParameter"}),
                         ("layer", 100, F.TYPE_MESSAGE, R, {"type_name": "LayerParameter"})])
    pool = descriptor_pool.DescriptorPool()
    pool.Add(fd)
    get = lambda n: message_factory.GetMessageClass(pool.FindMessageTypeByName("caffe_subset." + n))
    return get("NetParameter")


def _caffemodel_pb(layers: dict, mode: str) -> bytes:
    """mode: "shape" (BlobShape), "legacy" (num/channels/height/width, blob.cpp:448-462), "double" (double_data),
    "v1" (NetParameter.layers = V1LayerParameter, legacy dims)."""
    net = _caffe_pb()(name="net")
    for name, blobs in layers.items():
        lp = net.layers.add(name=name, type=4) if mode == "v1" else net.layer.add(name=name, type="Convolution")
        if mode != "v1":
            lp.bottom.append("x")
            lp.top.append(name)
        for b in blobs:
            bp = lp.blobs.add()
            if mode in ("legacy", "v1"):
                dims = [1] * (4 - b.ndim) + list(b.shape)     # legacy blobs index FROM THE END (blob.cpp:396-405)
                bp.num, bp.channels, bp.height, bp.width = dims
            else:
                bp.shape.dim.extend(b.shape)
            if mode == "double":
                bp.double_data.extend(b.astype(np.float64).reshape(-1).tolist())
            else:
                bp.data.extend(b.reshape(-1).tolist())
    return net.SerializeToString()


@pytest.mark.parametrize("encoder,mode", [("hand", "shape"), ("hand", "legacy"), ("pb", "shape"), ("pb", "legacy"),
                                          ("pb", "double"), ("pb", "v1")])
def test_caffemodel_wire_reader(tmp_path, encoder, mode):
    """Net::CopyTrainedLayersFrom(file) (net.cpp:787-803) through the library's own wire-format reader, against two
    independent encoders: the hand encoder above and the google.protobuf runtime; BlobShape and legacy 4-D dimensions
    (conv bias 1x1x1xN, InnerProduct weight 1x1xMxN: matched from the end of the shape, blob.cpp:392-413), double_data,
    and a V1 file (NetParameter.layers), which the reference upgrades on load."""
    from mscnn_b200.net import Net
    text = ('input: "data" input_dim: 1 input_dim: 64 input_dim: 6 input_dim: 6\n'
            'layer { bottom: "data" top: "c" name: "c" type: "Convolution" convolution_param { num_output: 8 kernel_size: 3 } }\n'
            'layer { bottom: "c" top: "f" name: "f" type: "InnerProduct" inner_product_param { num_output: 5 } }\n')
    rng = np.random.default_rng(5)
    w = {"c": [rng.standard_normal((8, 64, 3, 3)).astype(np.float32), rng.standard_normal(8).astype(np.float32)],
         "f": [rng.standard_normal((5, 128)).astype(np.float32), rng.standard_normal(5).astype(np.float32)],
         "not_in_net": [np.zeros((2, 2), np.float32)]}          # ignored like net.cpp:760-763
    path = tmp_path / "m.caffemodel"
    if encoder == "hand":
        legacy = mode == "legacy"
        wl = {k: [b.reshape((1,) * (4 - b.ndim) + b.shape) for b in v] for k, v in w.items()} if legacy else w
        path.write_bytes(_caffemodel(wl, legacy))
    else:
        path.write_bytes(_caffemodel_pb(w, mode))
    net = Net(text)
    net.copy_from(str(path))
    ref = Net(text)
    ref.set_params({k: v for k, v in w.items() if k != "not_in_net"})
    assert net.layer_param_strings() == ref.layer_param_strings()
    assert net.param_checksums() == ref.param_checksums()
    for name in ("c", "f"):
        for i, b in enumerate(w[name]):
            assert np.array_equal(net.param(name, i).reshape(-1), b.reshape(-1)), (name, i)


def test_caffemodel_truncated_file_is_rejected(tmp_path):
    """A file cut in the middle of a blob must abort like Caffe's ReadProtoFromBinaryFileOrDie (upgrade_proto.cpp),
    not read past the buffer; a file whose layers match nothing loads nothing and says so."""
    import subprocess
    import sys
    text = ('input: "data" input_dim: 1 input_dim: 64 input_dim: 6 input_dim: 6\n'
            'layer { bottom: "data" top: "c" name: "c" type: "Convolution" convolution_param { num_output: 8 kernel_size: 3 } }\n')
    w = {"c": [np.ones((8, 64, 3, 3), np.float32), np.ones(8, np.float32)]}
    full = _caffemodel_pb(w, "shape")
    bad = tmp_path / "cut.caffemodel"
    bad.write_bytes(full[: len(full) // 2])
    code = "import sys; from mscnn_b200.net import Net; n = Net(sys.argv[1]); n.copy_from(sys.argv[2])"
    root = str(Path(__file__).resolve().parents[1])
    r = subprocess.run([sys.executable, "-c", code, text, str(bad)], capture_output=True, text=True, cwd=root)
    assert r.returncode != 0 and "malformed caffemodel" in r.stderr
    other = tmp_path / "other.caffemodel"
    other.write_bytes(_caffemodel_pb({"zzz": [np.ones((2, 2), np.float32)]}, "shape"))
    r = subprocess.run([sys.executable, "-c", code, text, str(other)], capture_output=True, text=True, cwd=root)
    assert r.returncode == 0 and "none of its 1 layers matches" in r.stderr
