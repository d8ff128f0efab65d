"""Pins the CPU oracle (oracle.port) -- runs without a GPU.

 (a) the reference's own known-answer vectors for the upstream layers on the path, restated from
     /root/reference/src/caffe/test: pooling golden matrices (test_pooling_layer.cpp:49-119,
     543-573), the Sobel convolution identity (test_convolution_layer.cpp:498-589), the naive
     convolution loop the reference uses as ITS oracle (caffe_conv, :22-139), InnerProduct
     (test_inner_product_layer.cpp:107-139), Concat channels (test_concat_layer.cpp:143);
 (b) golden vectors generated from oracle/_ref = the reference's own layer code compiled verbatim
     (tests/golden/make_golden.py): BoxOutput and ROIPooling(pad_ratio), for which the reference
     ships no test at all;
 (c) port vs the reference build on seeded random inputs, bit-exact for the integer/ordering
     parts: the reference's outputs for those inputs are in tests/golden/port_vs_reference.npz
     (tests/golden/make_golden.py port).
"""
from pathlib import Path

import numpy as np
import pytest

from oracle import port

GOLD = Path(__file__).resolve().parent / "golden"


# ------------------------------------------------------------------ (a) upstream known answers
def test_pool_forward_square_golden():
    x = np.tile(np.array([[1, 2, 5, 2, 3], [9, 4, 1, 4, 8], [1, 2, 5, 2, 3]], dtype=np.float32), (2, 2, 1, 1))
    y = port.pool(x, kernel=2, stride=1, pad=0, mode="MAX")
    assert y.shape == (2, 2, 2, 4)
    assert np.array_equal(y[1, 1], np.array([[9, 5, 5, 8], [9, 5, 5, 8]], dtype=np.float32))


def test_pool_forward_ave_padded_golden():
    y = port.pool(np.full((1, 1, 3, 3), 2.0, dtype=np.float32), kernel=3, stride=1, pad=1, mode="AVE")
    exp = np.array([[8 / 9, 4 / 3, 8 / 9], [4 / 3, 2.0, 4 / 3], [8 / 9, 4 / 3, 8 / 9]])
    np.testing.assert_allclose(y[0, 0], exp, atol=1e-5)


def test_pool_ceil_mode_shape():
    # pooling_layer.cpp:90-93: ceil((H - k) / s) + 1
    assert port.pool(np.zeros((1, 1, 9, 15), np.float32), 2, 2).shape == (1, 1, 5, 8)
    assert port.pool(np.zeros((1, 1, 24, 80), np.float32), 2, 2).shape == (1, 1, 12, 40)


def _naive_conv(x, w, b, pad):
    n, c, h, wd = x.shape
    co, _, kh, kw = w.shape
    ho, wo = h + 2 * pad - kh + 1, wd + 2 * pad - kw + 1
    y = np.zeros((n, co, ho, wo), dtype=np.float64)
    for i in range(n):
        for o in range(co):
            for yy in range(ho):
                for xx in range(wo):
                    acc = 0.0
                    for k in range(c):
                        for p in range(kh):
                            for q in range(kw):
                                iy, ix = yy - pad + p, xx - pad + q
                                if 0 <= iy < h and 0 <= ix < wd:
                                    acc += float(x[i, k, iy, ix]) * float(w[o, k, p, q])
                    y[i, o, yy, xx] = acc + (float(b[o]) if b is not None else 0.0)
    return y


def test_conv_vs_naive_loops():
    rng = np.random.default_rng(1701)
    x = rng.standard_normal((2, 3, 6, 4)).astype(np.float32)     # the reference fixture shape
    w = rng.standard_normal((4, 3, 3, 3)).astype(np.float32)
    b = rng.standard_normal(4).astype(np.float32)
    np.testing.assert_allclose(port.conv2d(x, w, b, pad=1), _naive_conv(x, w, b, 1), atol=1e-4)
    w1 = rng.standard_normal((4, 3, 1, 1)).astype(np.float32)    # Test1x1Convolution
    np.testing.assert_allclose(port.conv2d(x, w1, b, pad=0), _naive_conv(x, w1, b, 0), atol=1e-4)


def test_conv_sobel_identity():
    """3x3 Sobel == (3x1 column [1 2 1]) o (1x3 row [-1 0 1]) (TestSobelConvolution)."""
    rng = np.random.default_rng(1702)
    x = rng.standard_normal((2, 1, 9, 8)).astype(np.float32)
    sobel = np.array([[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]], dtype=np.float32).reshape(1, 1, 3, 3)
    full = port.conv2d(x, sobel)
    col = port.conv2d(x, np.array([1, 2, 1], np.float32).reshape(1, 1, 3, 1))
    sep = port.conv2d(col, np.array([-1, 0, 1], np.float32).reshape(1, 1, 1, 3))
    np.testing.assert_allclose(full, sep, atol=1e-4)


def test_inner_product_and_concat():
    rng = np.random.default_rng(1703)
    x = rng.uniform(0, 1, (2, 3, 4, 5)).astype(np.float32)
    w = rng.uniform(0, 1, (10, 60)).astype(np.float32)
    b = rng.uniform(1, 2, 10).astype(np.float32)
    y = port.inner_product(x, w, b)
    assert y.shape == (2, 10) and (y >= 1).all()                 # TestForward: outputs >= 1
    np.testing.assert_allclose(y, x.reshape(2, -1).astype(np.float64) @ w.T.astype(np.float64) + b, rtol=1e-5)
    a, c = rng.standard_normal((2, 3, 4, 5)), rng.standard_normal((2, 2, 4, 5))
    cat = port.concat_channels(a, c)
    assert cat.shape == (2, 5, 4, 5) and np.array_equal(cat[:, 3:], c.astype(np.float32))


def test_box_iou_modes():
    assert port.box_iou((0, 0, 10, 10), (0, 0, 10, 10)) == 1.0
    assert port.box_iou((0, 0, 10, 10), (10, 0, 10, 10)) == 0.0          # touching: tlx >= brx
    assert port.box_iou((0, 0, 0, 10), (0, 0, 10, 10)) == 0.0            # degenerate width
    assert abs(port.box_iou((0, 0, 10, 10), (5, 0, 10, 10)) - 50.0 / 150.0) < 1e-7
    assert abs(port.box_iou((0, 0, 10, 10), (5, 0, 10, 5), "IOMU") - 25.0 / 50.0) < 1e-7
    assert abs(port.box_iou((0, 0, 10, 10), (5, 0, 10, 5), "IOFU") - 25.0 / 100.0) < 1e-7


def test_bilinear_filler_values():
    from mscnn_b200 import synth
    k = synth.bilinear_kernel(4)
    assert np.array_equal(k[0], np.array([0.0625, 0.1875, 0.1875, 0.0625], dtype=np.float32))
    x = np.ones((1, 2, 3, 3), np.float32)
    y = port.deconv_depthwise(x, np.broadcast_to(k, (2, 1, 4, 4)).copy())
    assert y.shape == (1, 2, 6, 6) and np.allclose(y[0, 0, 1:5, 1:5], 1.0)   # interior of an upsampled constant


# ---------------------------------------------------------------- (b) golden vectors from _ref
def test_box_output_golden():
    g = np.load(GOLD / "layers.npz")
    rois, sc, per, true = port.box_output([g["box_a"], g["box_b"]], [40, 80], [40, 80], [8, 16], fg_thr=-1.0,
                                          iou_thr=0.5, min_size=20.0, max_nms_num=40)
    assert np.array_equal(rois, g["box_rois"].reshape(-1, 5))
    assert np.array_equal(sc, g["box_rois_score"].reshape(-1, 6))
    assert true == len(rois) == per.sum()


def test_roi_pool_golden():
    g = np.load(GOLD / "layers.npz")
    assert np.array_equal(port.roi_pool(g["roi_x"], g["roi_r"], 7, 7, 0.125, 0.0), g["roi_org"])
    assert np.array_equal(port.roi_pool(g["roi_x"], g["roi_r"], 7, 7, 0.125, 0.25), g["roi_ctx"])


def test_box_output_empty_dummy_roi():
    m = np.zeros((1, 9, 4, 4), np.float32)
    m[:, 0] = 50.0
    rois, sc, per, true = port.box_output([m], [60], [60], [8], fg_thr=0.0, max_nms_num=10)
    assert true == 0 and rois.tolist() == [[0, 1, 1, 10, 10]] and not sc.any() and per.tolist() == [0]


def test_box_output_tie_break_prefers_larger_index():
    """std::greater<pair<score,idx>> (box_output_layer.cpp:168): equal scores -> later anchor first."""
    m = np.zeros((1, 9, 1, 3), np.float32)
    m[0, 1] = 3.0                           # identical scores at the three positions
    rois, sc, _, _ = port.box_output([m], [8], [8], [64], fg_thr=0.0, iou_thr=0.99, min_size=1.0, max_nms_num=10)
    assert len(rois) == 3 and rois[0, 1] > rois[1, 1] > rois[2, 1]


def test_detect_postprocess_basics():
    prop = np.array([[0, 10, 10, 110, 60, 5.0], [0, 12, 11, 112, 61, 4.0], [0, 500, 300, 560, 340, -20.0],
                     [0, 700, 100, 700, 150, 3.0]], dtype=np.float32)
    cls = np.zeros((4, 5), np.float32)
    cls[0, 1], cls[1, 1] = 3.0, 2.0
    bbox = np.zeros((4, 20), np.float32)
    det = port.detect_postprocess(prop, cls, bbox, cls_id=2, net_hw=(768, 2560))
    # row 2 dropped by the proposal threshold, row 3 by zero width, row 1 suppressed by row 0 (IoU > 0.5)
    assert det.shape == (1, 5)
    np.testing.assert_allclose(det[0, :4], [10, 10, 100, 50], atol=1e-4)
    assert abs(det[0, 4] - np.exp(3) / (np.exp(3) + 4)) < 1e-6


# --------------------------------------------------------------------- cascade-net layers
def test_cascade_layers_golden():
    """ROIAlign / DecodeBBox / Softmax / Eltwise restatements vs vectors generated from oracle/_ref
    (tests/golden/make_golden.py cascade): malformed, outside and sub-pixel ROIs, missing statistics,
    a saturating logit."""
    g = np.load(GOLD / "layers_cascade.npz")
    assert np.array_equal(port.roi_align(g["align_x"], g["align_r"], 5, 5, 0.125, 0.0), g["align_org"])
    assert np.array_equal(port.roi_align(g["align_x"], g["align_r"], 5, 5, 0.125, 0.25), g["align_ctx"])
    assert np.all(g["align_org"][1] == 0) and np.all(g["align_org"][2] == 0)   # malformed / outside -> zeros
    std = (0.05, 0.05, 0.1, 0.1)
    assert np.array_equal(port.decode_bbox(g["dec_b"], g["dec_p"], (0, 0, 0, 0), std), g["dec_out"].reshape(-1, 5))
    assert np.array_equal(port.decode_bbox(g["dec_b"], g["dec_p"]), g["dec_out_nostat"].reshape(-1, 5))
    sm = port.softmax(g["sm_x"])
    np.testing.assert_allclose(sm, g["sm_y"].reshape(6, 5), rtol=1e-6, atol=1e-12)
    np.testing.assert_allclose(sm.sum(1), 1.0, rtol=1e-6)
    sm_ref = g["sm_y"].reshape(6, 5)
    np.testing.assert_allclose(port.eltwise([g["sm_x"], sm_ref, g["sm_x"]], "SUM", [0.33333333, -2, 0.5]),
                               g["elt_sum"].reshape(6, 5), rtol=1e-6, atol=1e-7)
    assert np.array_equal(port.eltwise([g["sm_x"], sm_ref], "PROD"), g["elt_prod"].reshape(6, 5))
    assert np.array_equal(port.eltwise([g["sm_x"], sm_ref, g["elt_d1"]], "MAX"), g["elt_max"].reshape(6, 5))


@pytest.mark.parametrize("fixture,stds", [("e2e_cascade_kitti_96x320.npz", None), ("e2e_cascade_wider_128x192.npz", None)])
def test_cascade_stage_chain_golden(fixture, stds):
    """The stage-to-stage data flow of the cascade nets restated on the reference's own outputs:
    proposals_{k+1} = DecodeBBox(bbox_pred_k, proposals_k), cls_prob_k = Softmax(cls_pred_k)."""
    g = np.load(GOLD / fixture)
    stds = [(0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067)]
    pri = ["proposals", "proposals_2nd", "proposals_3rd"]
    bb = ["bbox_pred", "bbox_pred_2nd", "bbox_pred_3rd"]
    cp = ["cls_pred", "cls_pred_2nd", "cls_pred_3rd"]
    for k, nm in enumerate(["1st", "2nd", "3rd"]):
        r = len(g[pri[k]])
        dec = port.decode_bbox(g[bb[k]].reshape(r, -1), g[pri[k]], (0, 0, 0, 0), stds[k])
        assert np.array_equal(dec, g[f"output_bbox_{nm}"].reshape(r, 5))
        if k < 2:
            assert np.array_equal(dec, g[pri[k + 1]].reshape(r, 5))
        np.testing.assert_allclose(port.softmax(g[cp[k]].reshape(r, -1)), g[f"cls_prob_{nm}"].reshape(r, -1),
                                   rtol=2e-6, atol=1e-10)
    if "cls_prob_3rd_avg" in g:
        avg = port.eltwise([g["cls_prob_1st_3rd"], g["cls_prob_2nd_3rd"], g["cls_prob_3rd"]], "SUM", [0.33333333] * 3)
        np.testing.assert_allclose(avg, g["cls_prob_3rd_avg"], rtol=1e-6)


def test_cascade_detect_postprocess_basics():
    prop = np.array([[0, 10, 10, 109, 59], [0, 12, 11, 111, 60], [0, 700, 100, 699, 150], [0, 300, 200, 340, 260]],
                    dtype=np.float32)
    out = prop.copy()
    out[3] = [0, -20, 190, 2600, 900]       # clipped to the image
    prob = np.array([[0.1, 0.9], [0.3, 0.7], [0.2, 0.8], [0.6, 0.4]], dtype=np.float32)
    det = port.cascade_detect_postprocess(prop, prob, out, cls_id=2, net_hw=(768, 2560))
    # row 2 dropped (zero width: x2 - x1 + 1 == 0), row 1 suppressed by row 0
    assert det.shape == (2, 5)
    np.testing.assert_allclose(det[0], [10, 10, 100, 50, 0.9], atol=1e-6)
    np.testing.assert_allclose(det[1], [0, 190, 2561, 579, 0.4], atol=1e-6)


# ------------------------------------------------------ (c) port vs the verbatim reference build
def _box_output_case():
    """(deploy text, params by layer, input blobs, output blobs) of one reference run; make_golden.py port stores
    the reference's output blobs for it."""
    rng = np.random.default_rng(11)
    shapes = [(12, 40), (12, 40), (6, 20), (6, 20), (3, 10)]
    fields, rates = [60, 84, 120, 168, 240], [8, 8, 16, 16, 32]
    proto = "".join(f'input: "m{j}" input_dim: 2 input_dim: 9 input_dim: {h} input_dim: {w}\n'
                    for j, (h, w) in enumerate(shapes))
    proto += "layer { " + " ".join(f'bottom: "m{j}"' for j in range(5)) + ' top: "r" top: "rs" name: "p" type: "BoxOutput" '
    proto += 'box_output_param { fg_thr: -2 iou_thr: 0.65 nms_type: "IOU" ' + " ".join(f"field_w: {f} field_h: {f}" for f in fields)
    proto += " " + " ".join(f"downsample_rate: {r}" for r in rates) + " max_nms_num: 150 } }"
    blobs = {}
    for j, (h, w) in enumerate(shapes):
        m = rng.standard_normal((2, 9, h, w)).astype(np.float32)
        m[:, :5] *= 3
        m[:, 5:] *= 0.5
        blobs[f"m{j}"] = m
    return proto, {}, blobs, ["r", "rs"]


def _layers_case():
    rng = np.random.default_rng(12)
    proto = '''input: "x" input_dim: 2 input_dim: 16 input_dim: 9 input_dim: 11
layer { name: "c" type: "Convolution" bottom: "x" top: "c" convolution_param { num_output: 8 kernel_size: 5 pad: 2 } }
layer { name: "r" type: "ReLU" bottom: "c" top: "c" }
layer { name: "p" type: "Pooling" bottom: "c" top: "p" pooling_param { pool: MAX kernel_size: 2 stride: 2 } }
layer { name: "a" type: "Pooling" bottom: "c" top: "a" pooling_param { pool: AVE kernel_size: 2 stride: 2 } }
layer { name: "d" type: "Deconvolution" bottom: "c" top: "d" convolution_param { kernel_size: 4 stride: 2 num_output: 8 group: 8 pad: 1 weight_filler: { type: "bilinear" } bias_term: false } }
layer { name: "f" type: "InnerProduct" bottom: "p" top: "f" inner_product_param { num_output: 7 } }'''
    x = rng.standard_normal((2, 16, 9, 11)).astype(np.float32)
    w = rng.standard_normal((8, 16, 5, 5)).astype(np.float32) * 0.1
    b = rng.standard_normal(8).astype(np.float32)
    wf = rng.standard_normal((7, 8 * 5 * 6)).astype(np.float32) * 0.1
    bf = rng.standard_normal(7).astype(np.float32)
    return proto, {"c": [w, b], "f": [wf, bf]}, {"x": x}, ["c", "p", "a", "d", "f"]


def _cascade_layers_case():
    rng = np.random.default_rng(21)
    n, c, h, w, r = 2, 16, 14, 22, 60
    proto = f'''input: "x" input_dim: {n} input_dim: {c} input_dim: {h} input_dim: {w}
input: "r" input_dim: {r} input_dim: 5 input_dim: 1 input_dim: 1
input: "b" input_dim: {r} input_dim: 8 input_dim: 1 input_dim: 1
input: "s" input_dim: {r} input_dim: 5 input_dim: 3 input_dim: 2
layer {{ bottom: "x" bottom: "r" top: "a" name: "a" type: "ROIAlign" roi_pooling_param {{ pooled_w: 7 pooled_h: 4 spatial_scale: 0.25 pad_ratio: 0.125 }} }}
layer {{ bottom: "b" bottom: "r" top: "d" name: "d" type: "DecodeBBox" bbox_reg_param {{ bbox_mean: 0.1 bbox_mean: -0.1 bbox_mean: 0.05 bbox_mean: 0 bbox_std: 0.1 bbox_std: 0.1 bbox_std: 0.2 bbox_std: 0.2 }} }}
layer {{ bottom: "s" top: "sm" name: "sm" type: "Softmax" softmax_param {{ axis: 1 }} }}
layer {{ bottom: "s" top: "sl" name: "sl" type: "Softmax" softmax_param {{ axis: -1 }} }}'''
    x = rng.standard_normal((n, c, h, w)).astype(np.float32)
    x1 = rng.uniform(-10, 80, r); y1 = rng.uniform(-10, 50, r)
    rois = np.stack([rng.integers(0, n, r), x1, y1, x1 + rng.uniform(-5, 60, r), y1 + rng.uniform(-5, 40, r)], 1).astype(np.float32)
    b = rng.standard_normal((r, 8)).astype(np.float32)
    s = (rng.standard_normal((r, 5, 3, 2)) * 3).astype(np.float32)
    return proto, {}, {"x": x, "r": rois.reshape(r, 5, 1, 1), "b": b.reshape(r, 8, 1, 1), "s": s}, ["a", "d", "sm", "sl"]


PORT_CASES = {"box_output": _box_output_case, "layers": _layers_case, "cascade_layers": _cascade_layers_case}


def _reference(case):
    """The reference build's output blobs for PORT_CASES[case]."""
    g = np.load(GOLD / "port_vs_reference.npz")
    return {k.split("__", 1)[1]: g[k] for k in g.files if k.startswith(case + "__")}


def test_port_box_output_vs_reference_random():
    _, _, maps, _ = _box_output_case()
    ref = _reference("box_output")
    rois, sc, _, _ = port.box_output(list(maps.values()), [60, 84, 120, 168, 240], [60, 84, 120, 168, 240],
                                     [8, 8, 16, 16, 32], fg_thr=-2.0, iou_thr=0.65, max_nms_num=150)
    assert np.array_equal(rois, ref["r"].reshape(-1, 5))
    assert np.array_equal(sc, ref["rs"].reshape(-1, 6))


def test_port_layers_vs_reference_random():
    _, params, blobs, _ = _layers_case()
    (w, b), (wf, bf), x = params["c"], params["f"], blobs["x"]
    ref = _reference("layers")
    c = port.relu(port.conv2d(x, w, b, pad=2))
    np.testing.assert_allclose(c, ref["c"], rtol=1e-5, atol=1e-5)
    c = ref["c"]
    assert np.array_equal(port.pool(c, 2, 2), ref["p"])
    np.testing.assert_allclose(port.pool(c, 2, 2, mode="AVE"), ref["a"], rtol=1e-6)
    from mscnn_b200 import synth
    np.testing.assert_allclose(port.deconv_depthwise(c, np.broadcast_to(synth.bilinear_kernel(4), (8, 1, 4, 4)).copy()),
                               ref["d"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(port.inner_product(ref["p"], wf, bf), ref["f"], rtol=1e-5, atol=1e-5)


def test_port_cascade_layers_vs_reference_random():
    _, _, blobs, _ = _cascade_layers_case()
    x, s = blobs["x"], blobs["s"]
    r = len(blobs["r"])
    rois, b = blobs["r"].reshape(r, 5), blobs["b"].reshape(r, 8)
    ref = _reference("cascade_layers")
    assert np.array_equal(port.roi_align(x, rois, 4, 7, 0.25, 0.125)[::6], ref["a"])      # every 6th ROI stored
    assert np.array_equal(port.decode_bbox(b, rois, (0.1, -0.1, 0.05, 0), (0.1, 0.1, 0.2, 0.2)), ref["d"].reshape(r, 5))
    np.testing.assert_allclose(port.softmax(s, 1), ref["sm"], rtol=2e-6, atol=1e-10)
    np.testing.assert_allclose(port.softmax(s, 3), ref["sl"], rtol=2e-6, atol=1e-10)
