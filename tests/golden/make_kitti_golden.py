"""Regenerates tests/golden/kitti_eval/: the statistics files the REFERENCE evaluation tool
(examples/kitti_result/eval/evaluate_object.cpp, compiled verbatim by oracle/build_ref.py) writes for the seeded
synthetic label sets of tests/kitti_synth.py: seed 7 / 24 images (top level), seed 11 / 40 and seed 3 / 5 images
(seed11_n40/, seed3_n5/), and seed 21 / 16 images with oriented Car results only (orientation_seed21_n16/).  The
result files it reads are written by the product's mscnn_kitti_write_* entries (their formats are checked separately
in tests/test_kitti_eval.py).  `plot/<x>.txt` is stored as `plot_<x>.txt`.
Run where the reference tool has been built:  python tests/golden/make_kitti_golden.py"""
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(HERE.parent))

from kitti_synth import make_dataset, rows_to_padded, write_oriented_car_results  # noqa: E402
from mscnn_b200 import kitti  # noqa: E402

TOOL = ROOT / "oracle" / "_ref" / "evaluate_object"
OUT = HERE / "kitti_eval"
CASES = {(7, 24): OUT, (11, 40): OUT / "seed11_n40", (3, 5): OUT / "seed3_n5"}
ORIENTATION = (21, 16, OUT / "orientation_seed21_n16")


def _evaluate(td: Path, res: Path, out: Path) -> None:
    r = subprocess.run([str(TOOL), str(td / "label_2"), str(res), str(td / "val.txt")], capture_output=True, text=True)
    assert "done" in r.stdout, r.stdout + r.stderr
    out.mkdir(exist_ok=True)
    for f in res.glob("stats_*.txt"):
        shutil.copy(f, out / f.name)
    for f in (res / "plot").glob("*.txt"):
        shutil.copy(f, out / f"plot_{f.name}")


def main():
    for (seed, n), out in CASES.items():
        with tempfile.TemporaryDirectory() as td:
            td = Path(td)
            ids, rows = make_dataset(td, n_images=n, seed=seed)
            files = {}
            for cls, r in rows.items():
                dets, counts = rows_to_padded(r, n)
                files[cls] = td / f"{cls}.txt"
                kitti.write_det_file(files[cls], dets, counts)
            res = td / "res"
            kitti.write_labels(td / "val.txt", res / "data", car=files["Car"], ped=files["Pedestrian"], cyc=files["Cyclist"])
            _evaluate(td, res, out)
    seed, n, out = ORIENTATION
    with tempfile.TemporaryDirectory() as td:
        td = Path(td)
        ids, rows = make_dataset(td, n_images=n, seed=seed)
        write_oriented_car_results(td / "res", ids, rows)
        _evaluate(td, td / "res", out)
    print("wrote", sorted(str(p.relative_to(OUT)) for p in OUT.rglob("*.txt")))


if __name__ == "__main__":
    main()
