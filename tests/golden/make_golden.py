"""Generate the golden vectors under tests/golden/ from oracle/_ref -- the reference's own CPU
layer code compiled verbatim (oracle/build_ref.py).  Run where /root/reference is mounted:

    python tests/golden/make_golden.py

Outputs (committed):
  e2e_7s_192x640.npz   mscnn-7s-576 geometry, input 2x3x192x640 (synthetic seeded image + weights,
                       mscnn_b200/synth.py): the net outputs, all LFCN maps, the proposals, a fixed
                       subsample of conv4_3 / roi_c1 / fc6, per-blob second moments.
  e2e_7s2x_96x320.npz  mscnn-7s-576-2x geometry (Deconvolution + ROI scale 1/4), 1x3x96x320.
  layers.npz           single-layer known-answer vectors for BoxOutput / ROIPooling edge cases.
  e2e_cascade_kitti_96x320.npz   cascade-mscnn-7s-576-2x geometry, 2x3x96x320: per-stage proposals, class
                       probabilities, decoded boxes (`python tests/golden/make_golden.py cascade`).
  e2e_8s_192x640.npz   mscnn-8s-768 geometry (the bench architecture), 2x3x192x640 (main_8s).
  e2e_wider_128x192.npz  WIDER FACE mscnn-12s-2x geometry, 2x3x128x192 (main_wider).
  e2e_cascade_wider_128x192.npz  cascade-mscnn-12s-align geometry (ROIAlign, shared heads, Eltwise), 2x3x128x192.
  layers_cascade.npz   single-layer vectors for ROIAlign / DecodeBBox / Softmax / Eltwise edge cases.
  e2e_8s_768x2560.npz  mscnn-8s-768 at the BASELINE size (1x3x768x2560, configs[2]/[3]): every trunk blob incl.
                       conv3_1/3_2/3_3 and the pooled blobs sub-sampled (stride 1999), all eight LFCN maps, proposals,
                       head outputs (`python tests/golden/make_golden.py full`).
  e2e_wider_768x1024.npz  WIDER FACE mscnn-12s-2x at 1x3x768x1024 (configs[4]).
  e2e_7s2x_576x1920.npz   mscnn-7s-576-2x at 1x3x576x1920 (configs[1]).
  port_vs_reference.npz   the reference's output blobs for the seeded single-layer cases of tests/test_oracle.py
                       (`python tests/golden/make_golden.py port`).
  isolated_*.npz       the detection stages of mscnn-7s (1x3x96x320) and of both cascade nets fed with the reference's
                       own proposals and a seeded feature map (tests/test_net_gpu.py _synthetic_map): the proposals, the
                       map's scale and the stage outputs (every 16th row of the WIDER cascade; roi_c1 / fc6
                       sub-sampled) (`python tests/golden/make_golden.py isolated`).
  shipped_deploy_nets.json  sha256 digests of the structure of six of the reference's shipped deploy files as this
                       parser loads them (`python tests/golden/make_golden.py deploy`).
"""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
import numpy as np

from mscnn_b200 import models, synth
from oracle import ref

OUT = Path(__file__).resolve().parent
sys.path.insert(0, str(OUT.parent))
SUB = 7919  # subsample stride (prime)


def run_net(proto: str, n: int, h: int, w: int, keep: list[str], sub: list[str], SUB: int = SUB):
    net = ref.RefNet(proto, is_path=False)
    layers = [(nm, t, net.param_shapes(nm)) for nm, t in zip(net.layer_names, net.layer_types)]
    net.set_params(synth.make_weights(layers))
    net.set_blob("data", synth.make_images(n, h, w))
    net.forward()
    out = {}
    for b in keep:
        out[b] = net.blob(b)
    for b in sub:
        x = net.blob(b)
        out[b + "__sub"] = x.reshape(-1)[::SUB].copy()
        out[b + "__m2"] = np.array([np.mean(x.astype(np.float64) ** 2)], dtype=np.float64)
        out[b + "__shape"] = np.array(x.shape, dtype=np.int64)
    return out


def main():
    heads7 = ["LFCN_1_5x5", "LFCN_1_7x7", "LFCN_2_5x5", "LFCN_2_7x7", "LFCN_3_5x5", "LFCN_3_7x7", "LFCN_4_5x5"]
    g = run_net(models.kitti(192, 640, 7, False, batch=2), 2, 192, 640,
                keep=heads7 + ["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                sub=["conv1_2", "conv2_2", "conv3_3", "conv4_3", "conv5_3", "conv6_1", "roi_pool", "roi_c1", "fc6"])
    np.savez_compressed(OUT / "e2e_7s_192x640.npz", **g)
    print("e2e_7s_192x640: proposals", g["proposals"].shape)
    g = run_net(models.kitti(96, 320, 7, True, batch=1), 1, 96, 320,
                keep=["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                sub=["conv4_3", "conv4_3_2x", "roi_pool", "fc6"])
    np.savez_compressed(OUT / "e2e_7s2x_96x320.npz", **g)
    print("e2e_7s2x_96x320: proposals", g["proposals"].shape)

    # ---- single-layer vectors ---------------------------------------------------------------
    rng = np.random.default_rng(1706)
    vec = {}
    # BoxOutput: 2 scales, ties, clamps, border clipping, min_size
    box_proto = '''input: "a" input_dim: 2 input_dim: 9 input_dim: 6 input_dim: 10
input: "b" input_dim: 2 input_dim: 9 input_dim: 3 input_dim: 5
layer { bottom: "a" bottom: "b" top: "rois" top: "rois_score" name: "p" type: "BoxOutput"
  box_output_param { fg_thr: -1 iou_thr: 0.5 nms_type: "IOU" field_w: 40 field_w: 80 field_h: 40 field_h: 80
    downsample_rate: 8 downsample_rate: 16 field_whr: 2 field_xyr: 2 max_nms_num: 40 min_size: 20 } }'''
    net = ref.RefNet(box_proto, is_path=False)
    a = rng.standard_normal((2, 9, 6, 10)).astype(np.float32)
    b = rng.standard_normal((2, 9, 3, 5)).astype(np.float32)
    a[:, :5] = np.round(a[:, :5] * 2) / 2   # score ties
    b[:, :5] = np.round(b[:, :5] * 2) / 2
    a[:, 5:] *= 0.8
    b[:, 5:] *= 0.8
    net.set_blob("a", a)
    net.set_blob("b", b)
    net.forward()
    vec.update(box_a=a, box_b=b, box_rois=net.blob("rois"), box_rois_score=net.blob("rois_score"))
    # ROIPooling with pad_ratio: malformed / outside / half-pixel ROIs
    roi_proto = '''input: "x" input_dim: 2 input_dim: 8 input_dim: 12 input_dim: 20
input: "r" input_dim: 6 input_dim: 5 input_dim: 1 input_dim: 1
layer { bottom: "x" bottom: "r" top: "o" name: "o" type: "ROIPooling" roi_pooling_param { pooled_w: 7 pooled_h: 7 spatial_scale: 0.125 pad_ratio: 0 } }
layer { bottom: "x" bottom: "r" top: "c" name: "c" type: "ROIPooling" roi_pooling_param { pooled_w: 7 pooled_h: 7 spatial_scale: 0.125 pad_ratio: 0.25 } }'''
    net = ref.RefNet(roi_proto, is_path=False)
    x = rng.standard_normal((2, 8, 12, 20)).astype(np.float32)
    r = np.array([[0, 1, 1, 10, 10], [1, 50, 40, 30, 20], [0, 300, 300, 400, 400], [1, 3.5, 4.5, 4.5, 5.5],
                  [0, 0, 0, 159, 95], [1, 20.4, 11.6, 77.5, 60.5]], dtype=np.float32)
    net.set_blob("x", x)
    net.set_blob("r", r.reshape(6, 5, 1, 1))
    net.forward()
    vec.update(roi_x=x, roi_r=r, roi_org=net.blob("o"), roi_ctx=net.blob("c"))
    np.savez_compressed(OUT / "layers.npz", **vec)
    print("layers.npz:", {k: v.shape for k, v in vec.items()})


WIDER_HEADS = [f"LFCN_1_{z}x{z}" for z in (12, 16, 24, 32, 48)] + [f"LFCN_2_{z}x{z}" for z in (64, 96)] + \
    [f"LFCN_3_{z}x{z}" for z in (128, 192)] + [f"LFCN_4_{z}x{z}" for z in (256, 384, 480)]


def main_8s():
    """e2e_8s_192x640.npz: the bench architecture (mscnn-8s-768: eight heads, the last pair on pool6) at 2x3x192x640."""
    heads8 = [f"LFCN_{i}_{k}x{k}" for i in (1, 2, 3, 4) for k in (5, 7)]
    g = run_net(models.kitti(192, 640, 8, False, batch=2), 2, 192, 640,
                keep=heads8 + ["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                sub=["conv1_2", "conv2_2", "conv3_3", "conv4_3", "conv5_3", "conv6_1", "roi_pool", "fc6"])
    np.savez_compressed(OUT / "e2e_8s_192x640.npz", **g)
    print("e2e_8s_192x640: proposals", g["proposals"].shape)


def main_wider():
    """e2e_wider_128x192.npz: WIDER FACE mscnn-12s-2x geometry (twelve 1x1 heads of 6 channels, AVE pool6, bbox
    normalisation in BoxOutput, 5x5 ROI pooling on conv4_3_2x, fc6 2048), 2x3x128x192 (BASELINE.json configs[4])."""
    g = run_net(models.widerface(128, 192, batch=2), 2, 128, 192,
                keep=WIDER_HEADS + ["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                sub=["conv4_3", "conv4_3_2x", "conv5_3", "pool6", "roi_pool", "fc6"])
    np.savez_compressed(OUT / "e2e_wider_128x192.npz", **g)
    print("e2e_wider_128x192: proposals", g["proposals"].shape)


def main_cascade():
    stages = ["proposals", "proposals_2nd", "proposals_3rd", "output_bbox_1st", "output_bbox_2nd", "output_bbox_3rd",
              "cls_prob_1st", "cls_prob_2nd", "cls_prob_3rd", "cls_pred", "cls_pred_2nd", "cls_pred_3rd",
              "bbox_pred", "bbox_pred_2nd", "bbox_pred_3rd", "proposals_score"]
    g = run_net(models.kitti_cascade(96, 320, batch=2), 2, 96, 320, keep=stages,
                sub=["conv4_3_2x", "roi_pool", "roi_pool_2nd", "roi_pool_3rd", "fc6", "fc6_2nd", "fc6_3rd"])
    np.savez_compressed(OUT / "e2e_cascade_kitti_96x320.npz", **g)
    print("e2e_cascade_kitti_96x320: proposals", g["proposals"].shape)
    g = run_net(models.widerface_cascade(128, 192, batch=2), 2, 128, 192,
                keep=stages + ["cls_prob_1st_3rd", "cls_prob_2nd_3rd", "cls_prob_3rd_avg"],
                sub=["conv4_3", "roi_grid_org", "roi_grid_ctx", "roi_pool", "roi_pool_3rd", "fc6", "fc6_3rd",
                     "fc6_1st_3rd"])
    np.savez_compressed(OUT / "e2e_cascade_wider_128x192.npz", **g)
    print("e2e_cascade_wider_128x192: proposals", g["proposals"].shape)

    rng = np.random.default_rng(1707)
    vec = {}
    # ROIAlign: regular / malformed (x2 < x1) / outside the map / sub-pixel / whole-image ROIs, two pad ratios
    proto = '''input: "x" input_dim: 2 input_dim: 8 input_dim: 12 input_dim: 20
input: "r" input_dim: 7 input_dim: 5 input_dim: 1 input_dim: 1
layer { bottom: "x" bottom: "r" top: "o" name: "o" type: "ROIAlign" roi_pooling_param { pooled_w: 5 pooled_h: 5 spatial_scale: 0.125 pad_ratio: 0 } }
layer { bottom: "x" bottom: "r" top: "c" name: "c" type: "ROIAlign" roi_pooling_param { pooled_w: 5 pooled_h: 5 spatial_scale: 0.125 pad_ratio: 0.25 } }'''
    net = ref.RefNet(proto, is_path=False)
    x = rng.standard_normal((2, 8, 12, 20)).astype(np.float32)
    r = np.array([[0, 1, 1, 10, 10], [1, 50, 40, 30, 20], [0, 300, 300, 400, 400], [1, 3.5, 4.5, 4.5, 5.5],
                  [0, 0, 0, 159, 95], [1, 20.4, 11.6, 77.5, 60.5], [0, -30, -20, 40, 30]], dtype=np.float32)
    net.set_blob("x", x)
    net.set_blob("r", r.reshape(7, 5, 1, 1))
    net.forward()
    vec.update(align_x=x, align_r=r, align_org=net.blob("o"), align_ctx=net.blob("c"))
    # DecodeBBox + Softmax + Eltwise
    proto = '''input: "b" input_dim: 6 input_dim: 8 input_dim: 1 input_dim: 1
input: "p" input_dim: 6 input_dim: 5 input_dim: 1 input_dim: 1
input: "s" input_dim: 6 input_dim: 5
layer { name: "d" type: "DecodeBBox" bottom: "b" bottom: "p" top: "d" bbox_reg_param { bbox_mean: 0 bbox_mean: 0 bbox_mean: 0 bbox_mean: 0 bbox_std: 0.05 bbox_std: 0.05 bbox_std: 0.1 bbox_std: 0.1 } }
layer { name: "d0" type: "DecodeBBox" bottom: "b" bottom: "p" top: "d0" }
layer { name: "sm" type: "Softmax" bottom: "s" top: "sm" softmax_param { axis: 1 } }
layer { name: "es" type: "Eltwise" bottom: "s" bottom: "sm" bottom: "s" top: "es" eltwise_param { operation: SUM coeff: 0.33333333 coeff: -2 coeff: 0.5 } }
layer { name: "ep" type: "Eltwise" bottom: "s" bottom: "sm" top: "ep" eltwise_param { operation: PROD } }
layer { name: "em" type: "Eltwise" bottom: "s" bottom: "sm" bottom: "d1" top: "em" eltwise_param { operation: MAX } }'''
    proto = proto.replace('input: "s" input_dim: 6 input_dim: 5', 'input: "s" input_dim: 6 input_dim: 5 input_dim: 1 input_dim: 1\n'
                          'input: "d1" input_dim: 6 input_dim: 5 input_dim: 1 input_dim: 1')
    net = ref.RefNet(proto, is_path=False)
    b = (rng.standard_normal((6, 8)) * 2).astype(np.float32)
    p = np.array([[0, 10, 20, 50, 80], [1, 0, 0, 0, 0], [0, 100.5, 30.25, 90.5, 20.25], [1, -5, -5, 700, 300],
                  [0, 3, 4, 3, 4], [1, 17.3, 9.9, 64.2, 33.3]], dtype=np.float32)
    sc = (rng.standard_normal((6, 5)) * 4).astype(np.float32)
    sc[1] = 0          # uniform
    sc[2, 3] = 60      # saturating
    d1 = rng.standard_normal((6, 5)).astype(np.float32)
    net.set_blob("b", b.reshape(6, 8, 1, 1))
    net.set_blob("p", p.reshape(6, 5, 1, 1))
    net.set_blob("s", sc.reshape(6, 5, 1, 1))
    net.set_blob("d1", d1.reshape(6, 5, 1, 1))
    net.forward()
    vec.update(dec_b=b, dec_p=p, dec_out=net.blob("d"), dec_out_nostat=net.blob("d0"), sm_x=sc, sm_y=net.blob("sm"),
               elt_d1=d1, elt_sum=net.blob("es"), elt_prod=net.blob("ep"), elt_max=net.blob("em"))
    np.savez_compressed(OUT / "layers_cascade.npz", **vec)
    print("layers_cascade.npz:", {k: v.shape for k, v in vec.items()})


SUB_FULL = 1999
TRUNK_ALL = ["conv1_1", "conv1_2", "pool1", "conv2_1", "conv2_2", "pool2", "conv3_1", "conv3_2", "conv3_3", "pool3",
             "conv4_1", "conv4_2", "conv4_3", "pool4", "conv5_1", "conv5_2", "conv5_3", "pool5"]


def main_full(which=("8s", "wider", "7s2x")):
    """Full BASELINE sizes, one image each (one 768x2560 forward of the verbatim reference takes about a minute on
    8 cores).  Sub-sampling stride 1999 (prime; walks through every position class of every tiling)."""
    import time
    if "8s" in which:
        t = time.time()
        heads8 = [f"LFCN_{i}_{k}x{k}" for i in (1, 2, 3, 4) for k in (5, 7)]
        g = run_net(models.kitti(768, 2560, 8, False, batch=1), 1, 768, 2560,
                    keep=heads8 + ["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                    sub=TRUNK_ALL + ["conv6_1", "pool6", "loss1_conv1", "roi_pool", "roi_c1", "fc6"], SUB=SUB_FULL)
        np.savez_compressed(OUT / "e2e_8s_768x2560.npz", **g)
        print("e2e_8s_768x2560: proposals", g["proposals"].shape, f"{time.time() - t:.0f} s", flush=True)
    if "wider" in which:
        t = time.time()
        g = run_net(models.widerface(768, 1024, batch=1), 1, 768, 1024,
                    keep=WIDER_HEADS + ["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                    sub=TRUNK_ALL + ["conv4_3_2x", "pool6", "roi_pool", "roi_c1", "fc6"], SUB=SUB_FULL)
        np.savez_compressed(OUT / "e2e_wider_768x1024.npz", **g)
        print("e2e_wider_768x1024: proposals", g["proposals"].shape, f"{time.time() - t:.0f} s", flush=True)
    if "7s2x" in which:
        t = time.time()
        heads7 = ["LFCN_1_5x5", "LFCN_1_7x7", "LFCN_2_5x5", "LFCN_2_7x7", "LFCN_3_5x5", "LFCN_3_7x7", "LFCN_4_5x5"]
        g = run_net(models.kitti(576, 1920, 7, True, batch=1), 1, 576, 1920,
                    keep=heads7 + ["proposals", "proposals_score", "cls_pred", "bbox_pred"],
                    sub=TRUNK_ALL + ["conv6_1", "loss1_conv1", "conv4_3_2x", "roi_pool", "roi_c1", "fc6"], SUB=SUB_FULL)
        np.savez_compressed(OUT / "e2e_7s2x_576x1920.npz", **g)
        print("e2e_7s2x_576x1920: proposals", g["proposals"].shape, f"{time.time() - t:.0f} s", flush=True)


PORT_ALIGN_ROW_STEP = 6


def main_port():
    import test_oracle
    vec = {}
    for case, make in test_oracle.PORT_CASES.items():
        proto, params, blobs, outputs = make()
        net = ref.RefNet(proto, is_path=False)
        for layer, arrs in params.items():
            for k, a in enumerate(arrs):
                net.set_param(layer, k, a)
        for name, a in blobs.items():
            net.set_blob(name, a)
        net.forward()
        vec.update({f"{case}__{o}": net.blob(o) for o in outputs})
    vec["cascade_layers__a"] = vec["cascade_layers__a"][::PORT_ALIGN_ROW_STEP].copy()     # a fixed sample of the ROIs
    np.savez_compressed(OUT / "port_vs_reference.npz", **vec)
    print("port_vs_reference.npz:", {k: v.shape for k, v in vec.items()})


SUB_ISOLATED = 997
ROW_STEP = {"cascade_kitti": 1, "cascade_wider": 16}
CASCADE_STAGES = ["cls_pred", "bbox_pred", "proposals_2nd", "cls_pred_2nd", "bbox_pred_2nd", "proposals_3rd", "cls_pred_3rd",
                  "bbox_pred_3rd", "output_bbox_1st", "output_bbox_2nd", "output_bbox_3rd", "cls_prob_1st", "cls_prob_2nd",
                  "cls_prob_3rd"]


def main_isolated():
    """Each net runs once end to end for its proposals; then its feature map is replaced by the seeded stand-in (same
    shape, same second moment) and the stages after it run again."""
    from test_net_gpu import _isolated_protos, _synthetic_map
    for kind, (proto, (n, h, w), feat, first) in _isolated_protos().items():
        net = ref.RefNet(proto, is_path=False)
        layers = [(nm, t, net.param_shapes(nm)) for nm, t in zip(net.layer_names, net.layer_types)]
        net.set_params(synth.make_weights(layers))
        net.set_blob("data", synth.make_images(n, h, w))
        net.forward()
        real = net.blob(feat)
        scale = np.float64(np.sqrt(np.mean(real.astype(np.float64) ** 2) * 2))   # E[relu(z)^2] = 1/2
        fmap = _synthetic_map(real.shape, scale)
        net.set_blob(feat, fmap)             # the harness inserts no Split layers: every reader reads this blob
        net.forward(first)
        g = {"proposals": net.blob("proposals"), "fmap_scale": np.array([scale])}
        if kind == "head_7s":
            for b in ("cls_pred", "bbox_pred"):
                g[b] = net.blob(b)
            for b in ("roi_c1", "fc6"):
                x = net.blob(b)
                g[b + "__sub"] = x.reshape(-1)[::SUB_ISOLATED].copy()
                g[b + "__m2"] = np.array([np.mean(x.astype(np.float64) ** 2)])
                g[b + "__shape"] = np.array(x.shape, dtype=np.int64)
        else:
            # every row runs through the stages on its own: a fixed sample of the rows is stored
            g["rows"] = np.arange(0, len(g["proposals"]), ROW_STEP[kind])
            for b in CASCADE_STAGES + (["cls_prob_1st_3rd", "cls_prob_2nd_3rd", "cls_prob_3rd_avg"] if kind == "cascade_wider" else []):
                x = net.blob(b)
                g[b] = x[g["rows"]]
                g[b + "__shape"] = np.array(x.shape, dtype=np.int64)
        np.savez_compressed(OUT / f"isolated_{kind}.npz", **g)
        print(f"isolated_{kind}: proposals", g["proposals"].shape)


def main_deploy():
    """shipped_deploy_nets.json: the structure digests of the reference's shipped deploy files as this parser loads them."""
    import json
    from mscnn_b200.net import Net
    from oracle.build_ref import REF
    from test_net_cpu import SHIPPED_DEPLOY, net_structure
    out = {p: net_structure(Net(str(REF / "examples" / p / "mscnn_deploy.prototxt"))) for p, _ in SHIPPED_DEPLOY}
    (OUT / "shipped_deploy_nets.json").write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "full":
        main_full(tuple(sys.argv[2:]) or ("8s", "wider", "7s2x"))
    elif len(sys.argv) > 1 and sys.argv[1] == "cascade":
        main_cascade()
    elif len(sys.argv) > 1 and sys.argv[1] == "wider":
        main_wider()
    elif len(sys.argv) > 1 and sys.argv[1] == "8s":
        main_8s()
    elif len(sys.argv) > 1 and sys.argv[1] == "port":
        main_port()
    elif len(sys.argv) > 1 and sys.argv[1] == "isolated":
        main_isolated()
    elif len(sys.argv) > 1 and sys.argv[1] == "deploy":
        main_deploy()
    else:
        main()
        main_8s()
        main_wider()
        main_cascade()
