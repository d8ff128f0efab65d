"""Build oracle/_ref/libmscnn_ref.so: the reference's own CPU layer code, compiled VERBATIM
from the sources where they lie under /root/reference (never copied into this repo), against
the shim headers in oracle/ref_shim/ (glog / gflags / boost / cblas / caffe.pb.h stand-ins --
none of the real ones exist in the image), plus oracle/ref_harness.cpp.

TEST INFRASTRUCTURE ONLY.  Outputs go to oracle/_ref/ (git-ignored; travels to the GPU box
with the repo snapshot).  /root/reference does not exist on the GPU box, so this script is a
no-op there when the prebuilt library is present.

    python oracle/build_ref.py [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
REF = Path(os.environ.get("MSCNN_REFERENCE", "/root/reference"))
OUT = ROOT / "oracle" / "_ref"
LIB = OUT / "libmscnn_ref.so"
SHIM = ROOT / "oracle" / "ref_shim"

# Reference translation units on the MS-CNN forward path (SURVEY.md section 8(a)/(c)).
REF_SOURCES = [
    "src/caffe/common.cpp", "src/caffe/blob.cpp", "src/caffe/syncedmem.cpp", "src/caffe/layer.cpp",
    "src/caffe/util/math_functions.cpp", "src/caffe/util/im2col.cpp",
    "src/caffe/layers/neuron_layer.cpp", "src/caffe/layers/relu_layer.cpp",
    "src/caffe/layers/base_conv_layer.cpp", "src/caffe/layers/conv_layer.cpp",
    "src/caffe/layers/deconv_layer.cpp", "src/caffe/layers/pooling_layer.cpp",
    "src/caffe/layers/split_layer.cpp", "src/caffe/layers/concat_layer.cpp",
    "src/caffe/layers/inner_product_layer.cpp", "src/caffe/layers/dropout_layer.cpp",
    "src/caffe/layers/input_layer.cpp",
    "src/caffe/layers/box_output_layer.cpp", "src/caffe/layers/roi_pooling_layer.cpp",
    # cascade deploy nets (SURVEY.md section 8(f) rank 2)
    "src/caffe/layers/decode_bbox_layer.cpp", "src/caffe/layers/roi_align_layer.cpp",
    "src/caffe/layers/softmax_layer.cpp", "src/caffe/layers/eltwise_layer.cpp",
]
OWN_SOURCES = [SHIM / "cblas_shim.cpp", ROOT / "oracle" / "ref_harness.cpp"]

# -O2 without -march=native / -ffast-math: the reference Makefile's release flags
# (Makefile:318-322 "-DNDEBUG -O2"); keeps x86-64 baseline FP semantics (no FMA contraction).
CXXFLAGS = ["-std=c++14", "-O2", "-DNDEBUG", "-DCPU_ONLY", "-fPIC", "-fopenmp", "-w", "-fvisibility=hidden", "-fno-gnu-unique",
            "-I", str(SHIM), "-I", str(ROOT / "mscnn_b200" / "csrc" / "proto_shared"), "-I", str(REF / "include")]


def available() -> bool:
    return LIB.exists()


def present(p: Path) -> bool:
    """exists() that treats a reference tree this user may not read as absent (exists() raises on EACCES)."""
    try:
        return p.exists()
    except OSError:
        return False


KITTI_EVAL_SRC = REF / "examples" / "kitti_result" / "eval" / "evaluate_object.cpp"
KITTI_EVAL_BIN = OUT / "evaluate_object"


def build_kitti_eval(force: bool = False) -> Path | None:
    """The reference's KITTI evaluation tool (examples/kitti_result/eval/evaluate_object.cpp), a stand-alone
    program with no dependency beyond libstdc++: compiled verbatim from where it lies."""
    if not present(KITTI_EVAL_SRC):
        return KITTI_EVAL_BIN if KITTI_EVAL_BIN.exists() else None
    if KITTI_EVAL_BIN.exists() and not force and KITTI_EVAL_SRC.stat().st_mtime <= KITTI_EVAL_BIN.stat().st_mtime:
        return KITTI_EVAL_BIN
    OUT.mkdir(parents=True, exist_ok=True)
    r = subprocess.run(["g++", "-O2", "-w", "-o", str(KITTI_EVAL_BIN), str(KITTI_EVAL_SRC)], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed on evaluate_object.cpp:\n" + r.stderr[-4000:])
    return KITTI_EVAL_BIN


def build(force: bool = False) -> Path | None:
    build_kitti_eval(force)
    if not present(REF):
        return LIB if LIB.exists() else None
    srcs = [REF / s for s in REF_SOURCES] + OWN_SOURCES
    deps = srcs + list(SHIM.rglob("*.h*")) + list((ROOT / "mscnn_b200/csrc/proto_shared").rglob("*.h*")) + [Path(__file__)]
    if LIB.exists() and not force and all(d.stat().st_mtime <= LIB.stat().st_mtime for d in deps):
        return LIB
    obj = OUT / "obj"
    obj.mkdir(parents=True, exist_ok=True)

    def cc(src: Path) -> Path:
        o = obj / (src.stem + ".o")
        r = subprocess.run(["g++", *CXXFLAGS, "-c", str(src), "-o", str(o)], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"g++ failed on {src}:\n{r.stderr[-4000:]}")
        return o

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(cc, srcs))
    r = subprocess.run(["g++", "-shared", "-fopenmp", "-Wl,-Bsymbolic", "-o", str(LIB), *map(str, objs), "-ldl"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr[-4000:])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
