#!/usr/bin/env python
"""Benchmark of the MS-CNN detection forward path (BASELINE.json: images/sec, mscnn-8s-768
KITTI-car forward, batch 8 per B200, 3x768x2560 synthetic input; proposals/sec reported beside it).

    python bench.py --gpus 1 --steps K --warmup W            # this framework, one process per GPU
    torchrun --nproc-per-node N bench.py --gpus N ...        # image-parallel, weak scaling
    python bench.py --impl reference ...                     # the reference's CPU code on host cores

A "step" = one forward of one batch of 8 images per GPU through the whole path: conv trunk,
proposal heads, BoxOutput (decode + top-2000 + NMS), ROI pooling, detection head, final-detection
post-process; for N > 1 the post-process kernel also pushes the packed final detections into every rank's
gather buffer over NVLink (--exchange peer, default) or one ncclAllGather follows (--exchange nccl).

  value  : images/s, whole job, inputs already resident in HBM (fp32-faithful split-bf16 path, the
           path that meets the 1e-3 parity gate); `bf16` carries the same measurement for the plain
           bf16 tensor-core path (config 3 of BASELINE.json asks for both).
  e2e    : same metric through the public API (mscnn_b200.net.Net) with HOST buffers: pinned-host
           -> device copy of the batch and device -> host copy of the detections inside every step.
  roofline : the DOMINANT kernel instantiation (live CUDA-event times of the layers it serves); every instantiation in
           roofline.by_kernel; traffic from the committed ncu launch list of the current build.
  cpu_baseline / --impl reference : the reference's own CPU layers (oracle/_ref) on the SAME configuration, BLAS pinned to
           every host thread.  clocks / gpu_launches / per_rank_step_ms: see DESIGN.md section "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

NET_H, NET_W, BATCH = 768, 2560, 8
WORKLOAD = "mscnn-8s-768 KITTI-car forward, batch 8 per GPU, 3x768x2560 synthetic (BASELINE.json configs[2])"
CPU_SAMPLE_H, CPU_SAMPLE_W = 192, 640          # 1/16 of the pixels of one 768x2560 image


def peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))),
                "tflops_burst": float(d.get("bf16_tflops", 1590.0)), "hbm_gbs": float(d.get("hbm_gbs", 6650.0)),
                "source": "MEASURED_PEAKS.json (sustained cuBLAS bf16: kernel timed inside a long step)"}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median of the upper half = clocks while the GPU is loaded
        load = sm[len(sm) // 2:] if sm else []
        pw = sorted(float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "", 1).isdigit())
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": mx, "samples": len(sm),
                "power_w_max": (pw[-1] if pw else None), "reasons": sorted(reasons)}


def conv_flops(net, n_images: int) -> tuple[float, int]:
    """Algorithmic FLOPs of one forward (2*Cin*Cout*kh*kw*Hout*Wout*N per Convolution, 2*M*N*K per
    InnerProduct, SURVEY.md section 8(d)) using the shapes of the LAST forward (R is data dependent)."""
    total, launches = 0.0, 0
    for name, ltype, shapes in net.layers():
        if ltype == "Convolution":
            co, ci, kh, kw = shapes[0]
            n, _, ho, wo = net.blob_shape(name)
            total += 2.0 * ci * co * kh * kw * ho * wo * n
            launches += 1
        elif ltype == "InnerProduct":
            no, k = shapes[0]
            total += 2.0 * net.blob_shape(name)[0] * no * k
            launches += 1
    return total, launches


POOLED = ("conv1_2", "conv2_2", "conv3_3")     # 2x2 max pooling fused into the epilogue (never stored un-pooled)


def kernel_groups(net, layer_ms: dict, split: bool) -> list[dict]:
    """Per kernel instantiation: the Convolution / InnerProduct layers it serves in this net, their summed device
    time (CUDA events per layer) and algorithmic FLOPs.  The instantiation follows from the layer shape exactly as
    mscnn_conv_forward picks it (conv_igemm.cu pick_block_n / build_plan; pinned by tests/test_conv_plan_cpu.py):
    BLOCK_N = 256 | 128 | 64 | 32 by padded Cout; CTA pairs for the BLOCK_N = 256 layers of the fp32-faithful path;
    conv1_1 has its own kernel."""
    groups: dict[str, dict] = {}
    for name, ltype, shapes in net.layers():
        if ltype not in ("Convolution", "InnerProduct"):
            continue
        if ltype == "Convolution":
            co, ci, kh, kw = shapes[0]
            n, _, ho, wo = net.blob_shape(name)
            fl = 2.0 * ci * co * kh * kw * ho * wo * n
        else:
            co, k = shapes[0]
            ci, kh = k, 1
            fl = 2.0 * net.blob_shape(name)[0] * co * k
        if ltype == "Convolution" and ci == 3:
            kern, bound = "c3::conv_c3_tc_kernel", "hbm"
        elif ltype == "Convolution" and co in (6, 9) and kh > 1:
            kern, bound = "conv_igemm_kernel<64, false> (k x 1 head form) + head_gather_kernel", "tensor"
        else:
            cpad = (co + 63) // 64 * 64
            bn = 256 if cpad % 256 == 0 else 128 if cpad % 128 == 0 else 64
            pair = split and bn == 256 and co > 32      # un-pooled and pooled (conv3_3) BLOCK_N = 256 layers alike
            kern, bound = f"conv_igemm_kernel<{bn}, {'true' if pair else 'false'}>", "tensor"
        g = groups.setdefault(kern, {"kernel": kern, "bound": bound, "layers": [], "ms": 0.0, "gflop": 0.0})
        g["layers"].append(name)
        g["ms"] += layer_ms.get(name, 0.0)
        g["gflop"] += fl / 1e9
    out = sorted(groups.values(), key=lambda g: -g["ms"])
    for g in out:
        g["launches_per_step"] = len(g["layers"])
        g["tflops"] = g["gflop"] / max(g["ms"], 1e-9)
        g["ms"] = round(g["ms"], 3)
    return out


def launch_traffic(kernel: str):
    """Mean DRAM bytes per launch of `kernel` from the committed ncu launch list of the CURRENT build
    (profiles/r02_launches_summary.json, written by tools/summarize_launches.py); None when there is none."""
    p = ROOT / "profiles" / "r02_launches_summary.json"
    if not p.exists():
        return None, None
    d = json.loads(p.read_text())
    k = d["kernels"].get(kernel.replace(", ", ", ").split(" (")[0])
    if not k:
        return None, None
    return k["dram_read_bytes_per_launch"] + k["dram_write_bytes_per_launch"], f"profiles/r02_launches_summary.json ({d['source']}: mean over {k['launches']} launches of this instantiation)"


def _pin_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1; the reference arm is "all the host threads it can use"."""
    n = os.cpu_count() or 1
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = str(n)
    return n


def _ref_net(h: int, w: int):
    from oracle import ref
    from mscnn_b200 import models, synth
    net = ref.RefNet(models.kitti(h, w, 8, False, batch=1), is_path=False)
    layers = [(n, t, net.param_shapes(n)) for n, t in zip(net.layer_names, net.layer_types)]
    net.set_params(synth.make_weights(layers))
    net.set_blob("data", synth.make_images(1, h, w))
    return net


def _chunks(num_layers: int, k: int) -> list[list[tuple[int, int]]]:
    """K steps = n_full complete forwards, each cut into contiguous layer ranges [i0, i1] (inclusive)."""
    n_full = max(1, -(-k // num_layers))
    passes = []
    for p in range(n_full):
        c = k // n_full + (1 if p < k % n_full else 0)
        bounds = [round(j * num_layers / c) for j in range(c + 1)]
        passes.append([(bounds[j], bounds[j + 1] - 1) for j in range(c)])
    return passes


def run_reference(args) -> None:
    """--impl reference: the reference's own CPU implementation (oracle/_ref = its layer sources compiled verbatim),
    Caffe CPU mode, BLAS pinned to every host thread, on the SAME configuration as the GPU arm: real 3x768x2560 images
    through the full mscnn-8s net (so the ROI head is measured, not scaled by pixel count).  One such forward takes
    20-50 s on the box's cores, so a STEP is a bounded sample of it: the K timed steps are consecutive contiguous
    layer ranges that together make up exactly n_full = ceil(K / #layers) complete forwards of one image (K = 20 ->
    one forward in 20 slices); value = n_full images / total seconds.  Caffe's batch loop is per image
    (base_conv_layer.cpp:257-280 is called once per image, conv_layer.cpp:25-40), so images/s at batch 8 is the same
    figure.  Warm-up forwards run the 3x192x640 geometry (they page in the code and the BLAS threads)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = _pin_host_threads()
    from oracle import ref
    base = {"impl": "reference", "metric": "images/sec", "unit": "images/s", "higher_is_better": True,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "scaling": "weak", "dtype": "f32",
            "data": "synthetic", "vs_baseline": None,
            "config": {"workload": WORKLOAD, "global_batch": BATCH * args.gpus, "per_gpu_batch": BATCH,
                       "parallelism": f"dp{args.gpus}"}}
    if not ref.available():
        print(json.dumps({**base, "unavailable": "oracle/_ref/libmscnn_ref.so was not built (needs /root/reference at build time)"}))
        return
    cores = ref.set_blas_threads(ncpu)
    # tests/test_bench_cpu.py shrinks the image to exercise this arm in seconds; the line then says so in `config`
    full_h, full_w = NET_H, NET_W
    if os.environ.get("MSCNN_BENCH_TEST_HW"):
        full_h, full_w = (int(v) for v in os.environ["MSCNN_BENCH_TEST_HW"].split("x"))
        base["config"]["workload"] = f"TEST OVERRIDE {full_h}x{full_w} (not the benchmark workload)"
    small = _ref_net(min(CPU_SAMPLE_H, full_h), min(CPU_SAMPLE_W, full_w))
    for _ in range(max(1, min(args.warmup, 2))):
        small.forward()
    del small
    net = _ref_net(full_h, full_w)
    names = net.layer_names
    passes = _chunks(len(names), max(1, args.steps))
    step_s = []
    t_all = time.perf_counter()
    for chunks in passes:
        for i0, i1 in chunks:
            t0 = time.perf_counter()
            net.forward(names[i0], names[i1])
            step_s.append(time.perf_counter() - t0)
    total = time.perf_counter() - t_all
    n_full = len(passes)
    value = n_full / total
    rows = int(net.blob_shape("proposals")[0])
    sample = (f"{n_full} complete forward(s) of 1 synthetic 3x{full_h}x{full_w} image through the full mscnn-8s net (R = {rows} "
              f"proposals), cut into {len(step_s)} consecutive layer-range steps; Caffe CPU mode, reference layers compiled "
              f"verbatim, {ref.blas_backend()}, {cores} BLAS threads of {ncpu} host cpus; images/s = {n_full} / {total:.1f} s")
    line = {**base, "value": value, "ms_per_step": total / len(step_s) * 1e3,
            "seconds_per_image": total / n_full, "proposals_per_image": rows,
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def cpu_baseline() -> dict:
    """The reference's CPU path on the box's host cores, same configuration: ONE complete forward of one real
    3x768x2560 image (20-50 s), after a warm-up forward of the 3x192x640 geometry."""
    ncpu = _pin_host_threads()
    from oracle import ref
    if not ref.available():
        return {"value": None, "unit": "images/s", "cores": 0, "kind": "reference",
                "sample": "oracle/_ref not built on this machine"}
    cores = ref.set_blas_threads(ncpu)
    small = _ref_net(CPU_SAMPLE_H, CPU_SAMPLE_W)
    small.forward()                     # warm-up forward (caffe time does one, tools/caffe.cpp:359-362)
    del small
    net = _ref_net(NET_H, NET_W)
    t0 = time.perf_counter()
    per_layer = net.forward()
    dt = time.perf_counter() - t0
    top = sorted(per_layer.items(), key=lambda kv: -kv[1])[:5]
    return {"value": 1.0 / dt, "unit": "images/s", "cores": cores, "kind": "reference",
            "sample": (f"1 forward of 1 synthetic 3x{NET_H}x{NET_W} image (= 1/{BATCH} of a step) through the full mscnn-8s "
                       f"net with the reference's own CPU layers (compiled verbatim, Caffe CPU mode, {ref.blas_backend()}, "
                       f"{cores} BLAS threads of {ncpu} host cpus): {dt:.1f} s"),
            "seconds_per_image": dt, "top_layers_s": [[k, round(v / 1e3, 2)] for k, v in top]}


def parallel_first_index(rank: int, per_gpu_batch: int) -> int:
    from mscnn_b200 import parallel
    return parallel.shard_range(rank, per_gpu_batch)[0]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mscnn_b200", choices=["mscnn_b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bf16", action="store_true", help="skip the plain-bf16 measurement")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: 'peer' = the post-process kernel pushes its payload into every rank's buffer over NVLink "
                         "(no collective kernel; default); 'nccl' = one ncclAllGather per step on a side stream (baseline)")
    ap.add_argument("--generations", type=int, default=16,
                    help="peer exchange: how many steps the ranks may drift apart (2 = meet every step)")
    ap.add_argument("--no-gather", action="store_true",
                    help="control run for the scaling analysis: N > 1 without the all-gather of the final detections")
    ap.add_argument("--resident-only", action="store_true", help="only the device-resident measurement (no e2e loops)")
    ap.add_argument("--profile-bf16", action="store_true",
                    help="profiling aid: run ONLY plain-bf16 forwards and print nothing (for ncu captures)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step (fp32, inputs resident) returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "mscnn_b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from mscnn_b200 import capi, models, net as mnet, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its banner ("NCCL version ...") to stdout when NCCL_DEBUG >= VERSION: keep stdout = the JSON line
        # (NCCL honours NCCL_DEBUG_FILE only above the VERSION level, so VERSION is raised to WARN)
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    mnet.set_device(local)
    mnet.set_stream(torch.cuda.current_stream().cuda_stream)
    B = args.batch

    net = mnet.Net(models.kitti(NET_H, NET_W, 8, False, batch=B))
    net.set_params(synth.make_weights(net.layers()))
    first = parallel_first_index(rank, B)
    host_img = torch.from_numpy(synth.make_images(B, NET_H, NET_W, first_index=first)).pin_memory()
    dev_img = host_img.to(dev, non_blocking=True)
    cfg = mnet.kitti_detect_cfg(NET_H, NET_W)
    cap = cfg.max_rois_per_image
    dets = torch.zeros((B, cap, 5), device=dev)
    cnt = torch.zeros(B, dtype=torch.int32, device=dev)
    host_dets = torch.zeros((B, cap, 5)).pin_memory()
    host_cnt = torch.zeros(B, dtype=torch.int32).pin_memory()
    from mscnn_b200 import parallel
    # N > 1: the path's only exchange (SURVEY.md 8(e)) lives in the C++ library: final detections packed on the device
    # (per-image counts in the payload header) + ONE ncclAllGather on the communicator's own stream, overlapping the
    # next step's trunk (mscnn_net_detect_gather).  torch.distributed only carries the NCCL id and the barriers.
    use_gather = world > 1 and not args.no_gather
    use_peer = use_gather and args.exchange == "peer"
    comm = parallel.Comm() if (use_gather and not use_peer) else None
    per = parallel.payload_floats(B, cap)
    xchg = parallel.PeerExchange(B, cap, generations=args.generations) if use_peer else None
    exchange_note = None
    if use_peer and not xchg.ok:       # peer mapping unavailable on this box: every rank falls back to NCCL together
        exchange_note = f"peer-memory exchange unavailable ({xchg.error}); fell back to --exchange nccl"
        xchg, use_peer = None, False
        comm = parallel.Comm()
    payload_all = torch.zeros(per * world, device=dev) if (use_gather and not use_peer) else None
    host_payload = torch.zeros(per).pin_memory() if use_gather else None
    cur_stream = torch.cuda.current_stream().cuda_stream

    def detect():
        if use_peer:
            net.detect_push(cfg, xchg)          # post-process + push to every rank + flags: ONE set of kernels
        elif use_gather:
            net.detect_gather(cfg, comm, payload_all.data_ptr())
        else:
            net.detect(cfg, dets.data_ptr(), cnt.data_ptr())

    def download():
        # device -> host read of this rank's result (its own packed detections when the exchange is on)
        if use_peer:
            host_payload.copy_(xchg.gathered()[rank * per:(rank + 1) * per], non_blocking=True)
        elif use_gather:
            host_payload.copy_(payload_all[rank * per:(rank + 1) * per], non_blocking=True)
        else:
            host_dets.copy_(dets, non_blocking=True)
            host_cnt.copy_(cnt, non_blocking=True)

    def step_resident():
        net.set_input("data", dev_img)          # D2D into the net's input blob (inputs resident in HBM)
        net.forward_only()
        detect()

    def step_e2e_serial():
        net.set_input("data", host_img)         # pinned host -> device, async on the net stream
        net.forward_only()
        detect()
        download()
        torch.cuda.current_stream().synchronize()

    def step_e2e():
        # Software-pipelined over steps, as a throughput deployment feeds the net: every step still does one
        # H2D upload of a full input batch from pinned host memory and one D2H read of its detections, but the
        # upload is the NEXT step's input, issued on the copy stream as soon as this step's forward has been
        # queued (it starts on the device once conv1_1 of this step has consumed the blob), so it overlaps the
        # ROI head instead of preceding the trunk.  The first timed step's input was uploaded by the last
        # warm-up step; K timed steps contain exactly K uploads and K downloads.
        net.forward_only()
        detect()
        net.set_input_async("data", host_img)
        download()
        torch.cuda.current_stream().synchronize()

    # the MATLAB driver's own entry: ORIGINAL uint8 frames (KITTI: 375 x 1242) -> imresize + BGR + mean + CHW on
    # the device -> forward -> detections (SURVEY.md 8(f)-3); 11 MB of H2D per step instead of 189 MB
    from mscnn_b200 import ops as mops
    ORG_H, ORG_W = 375, 1242
    pre = mops.Preprocess((ORG_H, ORG_W), (NET_H, NET_W))
    rng_u8 = np.random.default_rng(1706 + first)
    host_u8 = torch.from_numpy(rng_u8.integers(0, 256, size=(B, ORG_H, ORG_W, 3), dtype=np.uint8)).pin_memory()

    def step_e2e_images():
        net.set_input_images("data", pre, host_u8)
        net.forward_only()
        detect()
        download()
        torch.cuda.current_stream().synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        n0 = capi.lib().mscnn_kernel_launch_count()
        ev[0].record()
        for i in range(steps):
            fn()
            ev[i + 1].record()
        if use_peer:
            xchg.wait(cur_stream)               # the timed region ends when every rank's last payload has landed here
        elif use_gather:
            comm.stream_wait(cur_stream)        # the timed region ends when the last step's all-gather has landed
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        torch.cuda.synchronize()
        launched = capi.lib().mscnn_kernel_launch_count() - n0
        timed.step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        if world > 1:
            dist.barrier()
        ms = torch.tensor([ev[0].elapsed_time(e1), float(launched)], device=dev)
        if world > 1:
            both = ms.clone()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(both, op=dist.ReduceOp.SUM)
            ms[1] = both[1]
        timed.launched = int(ms[1].item())     # kernels launched by libmscnn_b200 in the timed region, all ranks
        return float(ms[0].item())

    if args.profile_bf16:
        mnet.set_precision("bf16")
        for _ in range(args.warmup + args.steps):
            step_resident()
        torch.cuda.synchronize()
        return

    def outputs() -> dict:
        """What a caller of the timed path receives: the net's outputs and the final detections (or, with the
        exchange on, the gathered payload of every rank), as float32 / float64 arrays."""
        out = {name: net.blob(name).astype(np.float32) for name in net.outputs}
        if use_peer:
            out["gathered_payload"] = xchg.gathered().cpu().numpy().astype(np.float32)
        elif use_gather:
            out["gathered_payload"] = payload_all.cpu().numpy().astype(np.float32)
        else:
            out["detections"] = dets.cpu().numpy().astype(np.float32)
            out["detection_counts"] = cnt.cpu().numpy().astype(np.float64)
        return out

    results = {}
    dumped = None
    sampler = ClockSampler(local)      # every rank samples ITS GPU: the scaling analysis needs the slowest one's clocks
    for mode in (["fp32"] if args.no_bf16 else ["fp32", "bf16"]):
        mnet.set_precision(mode)
        if mode == "fp32" and sampler:
            sampler.start()
        ms = timed(step_resident, args.steps, args.warmup)
        launched = timed.launched
        if mode == "fp32" and args.dump_outputs and rank == 0:
            dumped = outputs()
        step_ms = sorted(timed.step_ms)
        clocks = sampler.stop() if (mode == "fp32" and sampler) else None
        per_rank = None
        if world > 1 and mode == "fp32":
            # where the time goes at N > 1: each rank's own step times (device events between steps on ITS stream)
            mine = {"rank": rank, "min": round(step_ms[0], 3), "median": round(step_ms[len(step_ms) // 2], 3),
                    "max": round(step_ms[-1], 3), "sum": round(sum(step_ms), 3)}
            mine["sm_mhz"] = clocks["sm_mhz"] if clocks else None
            mine["power_w_max"] = clocks.get("power_w_max") if clocks else None
            mine["reasons"] = clocks["reasons"] if clocks else None
            if use_gather and not use_peer:
                gt = sorted(comm.gather_times_ms(min(args.steps, 64)))
                mine["gather_ms"] = {"min": round(gt[0], 4), "median": round(gt[len(gt) // 2], 4), "max": round(gt[-1], 4)}
            per_rank = [None] * world
            dist.all_gather_object(per_rank, mine)
        props = torch.tensor([float(net.num_proposals())], device=dev)
        if world > 1:
            dist.all_reduce(props)
        if args.resident_only:
            ms_e2e_serial = ms_e2e = ms_e2e_images = float("nan")
        else:
            ms_e2e_serial = timed(step_e2e_serial, args.steps, args.warmup)
            net.set_input_async("data", host_img)   # prologue of the pipelined loop
            ms_e2e = timed(step_e2e, args.steps, args.warmup)
            ms_e2e_images = timed(step_e2e_images, args.steps, args.warmup) if mode == "fp32" else None
        net.set_input("data", dev_img)
        # per-layer device times for the roofline: two extra forwards with CUDA events per layer
        mnet.set_precision(mode)
        lt = net.time_layers()
        lt2 = net.time_layers()
        types = dict(zip(net.layer_names, net.layer_types))
        conv_ms = sum(min(lt[k], lt2[k]) for k in lt if types[k] in ("Convolution", "InnerProduct"))
        all_ms = sum(min(lt[k], lt2[k]) for k in lt)
        flops, conv_launches = conv_flops(net, B)
        by_kernel = kernel_groups(net, {k: min(lt[k], lt2[k]) for k in lt}, mode == "fp32")
        results[mode] = dict(by_kernel=by_kernel, per_rank=per_rank, ms=ms, ms_e2e=ms_e2e, ms_e2e_serial=ms_e2e_serial, ms_e2e_images=ms_e2e_images, props=float(props.item()), conv_ms=conv_ms, all_ms=all_ms,
                             flops=flops, conv_launches=conv_launches, clocks=clocks, launched=launched,
                             top=sorted(((min(lt[k], lt2[k]), k) for k in lt), reverse=True)[:6],
                             layers={k: round(min(lt[k], lt2[k]), 3) for k in lt if min(lt[k], lt2[k]) >= 0.02})
    mnet.set_precision("fp32")

    if comm is not None:
        comm.synchronize()
        comm.close()
    if xchg is not None:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()                      # nobody unmaps a buffer a peer may still be writing
        xchg.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if dumped is not None:
        d = Path(args.dump_outputs)
        d.mkdir(parents=True, exist_ok=True)
        for name, a in dumped.items():
            np.save(d / f"{name}.npy", a)
    pk = peaks()

    def roofline(r, pk):
        """Top level = the DOMINANT kernel instantiation (largest share of the step): achieved = its layers'
        algorithmic FLOPs / their summed CUDA-event time, measured live; `by_kernel` holds every instantiation with
        its own fraction; `all_conv_fc` is the lumped figure earlier rounds reported."""
        dom = next(g for g in r["by_kernel"] if g["bound"] == "tensor")
        traffic, tsrc = launch_traffic(dom["kernel"])
        ach_all = r["flops"] / (r["conv_ms"] / 1e3) / 1e12
        by = []
        for g in r["by_kernel"]:
            e = {"kernel": g["kernel"], "bound": g["bound"], "layers": g["layers"], "ms_per_step": g["ms"],
                 "share_of_step": round(g["ms"] / r["all_ms"], 4), "algorithmic_gflop_per_step": round(g["gflop"], 1),
                 "achieved_tflops": round(g["tflops"], 1), "frac_of_tensor_peak": round(g["tflops"] / pk["tflops"], 4)}
            if g["bound"] == "hbm":
                # conv1_1: 12 B in + 256 B out per pixel (fp32 NCHW image in, (hi, lo) planes of 64 channels out)
                gb = B * NET_H * NET_W * (12 + 256) / 1e9
                e["algorithmic_gb_per_step"] = round(gb, 3)
                e["achieved_gbs"] = round(gb / (g["ms"] / 1e3), 1)
                e["frac_of_hbm_peak"] = round(e["achieved_gbs"] / pk["hbm_gbs"], 4)
            by.append(e)
        return {"bound": "tensor", "kernel": dom["kernel"], "layers": dom["layers"],
                "achieved": dom["tflops"], "peak": pk["tflops"], "unit": "TFLOP/s", "frac": dom["tflops"] / pk["tflops"],
                "traffic": traffic, "traffic_source": tsrc,
                "algorithmic_gflop_per_launch": dom["gflop"] / dom["launches_per_step"],
                "launches_per_step": dom["launches_per_step"],
                "avg_launch_ms": dom["ms"] / dom["launches_per_step"],
                "share_of_step": dom["ms"] / r["all_ms"],
                "executed_tensor_flops_factor": 3,
                "frac_executed": 3 * dom["tflops"] / pk["tflops"],
                "peak_source": pk["source"],
                "how": "algorithmic FLOPs (2 Cin Cout kh kw Ho Wo N; 2 M N K) of the layers this instantiation serves / "
                       "the sum of their per-layer CUDA-event times (two timed forwards after the timed region, min per "
                       "layer, same stream); the fp32-faithful path executes 3 bf16 products per algorithmic FLOP, so "
                       "frac <= 1/3 and frac_executed = 3 frac is the tensor-pipe view",
                "by_kernel": by,
                "all_conv_fc": {"achieved": ach_all, "frac": ach_all / pk["tflops"],
                                "algorithmic_gflop_per_step": r["flops"] / 1e9, "launches_per_step": r["conv_launches"],
                                "share_of_step": r["conv_ms"] / r["all_ms"]}}

    r = results["fp32"]
    total_images = B * world * args.steps
    value = total_images / (r["ms"] / 1e3)
    e2e_value = total_images / (r["ms_e2e"] / 1e3)
    achieved = r["flops"] / (r["conv_ms"] / 1e3) / 1e12
    line = {
        "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms"] / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16x3 (fp32-faithful: 3-term bf16 split on tcgen05, fp32 accumulate in TMEM)",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": B * world, "per_gpu_batch": B,
                   "parallelism": (f"dp{world} image-parallel" + (
                       ", final detections pushed into every rank's buffer over NVLink by the post-process kernel itself "
                       "(peer-mapped stores + flags, no collective kernel)" if use_peer else
                       ", one ncclAllGather of the packed final detections per step inside libmscnn_b200.so (side stream)"
                       if use_gather else (", exchange OFF (--no-gather control run)" if world > 1 else ""))),
                   "l2": "inputs larger than L2 (189 MB image batch + >10 GB of activations per step vs 126 MB L2)",
                   "weights": "seeded synthetic (mscnn_b200/synth.py), seed 1706"},
        "proposals_per_sec": r["props"] * args.steps / (r["ms"] / 1e3),
        "proposals_per_image": r["props"] / (B * world),
        "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": r["ms_e2e"] / args.steps,
                "h2d_bytes_per_step": B * 3 * NET_H * NET_W * 4 * world,
                "d2h_bytes_per_step": (per * 4 if use_gather else B * cap * 5 * 4 + B * 4) * world,
                "pipelined": True,   # the upload inside step k is step k+1's batch; serial_* below is the strict order
                "serial_value": total_images / (r["ms_e2e_serial"] / 1e3),
                "serial_ms_per_step": r["ms_e2e_serial"] / args.steps,
                "api": "mscnn_b200.net.Net: forward_only / detect / set_input_async(pinned host, next step's batch, "
                       "copy stream) / D2H of detections + sync, software-pipelined over steps (one full-batch upload "
                       "and one download inside every timed step); serial_* = set_input / forward / detect / D2H "
                       "strictly in order on one stream"},
        # same loop fed with ORIGINAL uint8 frames: upload + device pre-processing (imresize bicubic/antialias, BGR,
        # mean, CHW) + forward + detect + download, strictly serial on the net stream (random uint8 frames, so the
        # proposal count differs from the headline workload)
        "e2e_images": {"value": total_images / ((r["ms_e2e_images"] or float("nan")) / 1e3), "unit": "images/s",
                       "ms_per_step": (r["ms_e2e_images"] or float("nan")) / args.steps,
                       "h2d_bytes_per_step": B * 375 * 1242 * 3 * world,
                       "d2h_bytes_per_step": (B * cap * 5 * 4 + B * 4) * world,
                       "api": "Net.set_input_images(uint8 375x1242 frames, ops.Preprocess) / forward_only / detect / D2H"},
        # counted by the library itself (mscnn_kernel_launch_count) inside the timed resident region, all ranks
        "gpu_launches": r["launched"],
        "roofline": roofline(r, pk),
        "clocks": r["clocks"],
        "exchange": ("off" if not use_gather else "peer" if use_peer else "nccl") + (f" ({exchange_note})" if exchange_note else ""),
        "per_rank_step_ms": r["per_rank"],
        "top_layers_ms": [[k, round(v, 3)] for v, k in r["top"]],
        "layers_ms": r["layers"],
    }
    if "bf16" in results:
        b = results["bf16"]
        ach_b = b["flops"] / (b["conv_ms"] / 1e3) / 1e12
        line["bf16"] = {"value": total_images / (b["ms"] / 1e3), "unit": "images/s", "ms_per_step": b["ms"] / args.steps,
                        "e2e_value": total_images / (b["ms_e2e"] / 1e3),
                        "e2e_serial_value": total_images / (b["ms_e2e_serial"] / 1e3),
                        "roofline": {"achieved": ach_b, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach_b / pk["tflops"]},
                        "note": "plain bf16 conv path: fails the 1e-3 parity gate (bf16 rounding of activations), "
                                "reported as BASELINE.json config 3 asks; proposals/image differ accordingly",
                        "proposals_per_image": b["props"] / (B * world),
                        "top_layers_ms": [[k, round(v, 3)] for v, k in b["top"]], "layers_ms": b["layers"]}
    if args.resident_only:          # control runs (scaling analysis): no end-to-end loops were timed
        line.pop("e2e")
        line.pop("e2e_images")
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
