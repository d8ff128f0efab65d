"""KITTI result writer / evaluator glue (SURVEY.md 8(f)-4), host-only C-ABI entries mscnn_kitti_*.

Oracle: the reference's own tool examples/kitti_result/eval/evaluate_object.cpp compiled VERBATIM
(oracle/build_ref.py -> oracle/_ref/evaluate_object).  The statistics files it wrote for seeded synthetic label sets
are committed under tests/golden/kitti_eval/ (tests/golden/make_kitti_golden.py), and the files of this evaluator are
compared with them byte for byte.  The two MATLAB writer steps (dlmwrite / writeLabels record formats) are restated
from the scripts and are parity-unpinned beyond the format checks below."""
from pathlib import Path

import numpy as np
import pytest

from kitti_synth import make_dataset, rows_to_padded, write_oriented_car_results

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = Path(__file__).resolve().parent / "golden" / "kitti_eval"
GOLDEN_CASES = {(7, 24): ".", (11, 40): "seed11_n40", (3, 5): "seed3_n5"}


def _write_results(root, rows, n_images, comp="res"):
    from mscnn_b200 import kitti
    files = {}
    for cls, r in rows.items():
        dets, counts = rows_to_padded(r, n_images)
        files[cls] = root / f"{comp}_{cls.lower()}.txt"
        kitti.write_det_file(files[cls], dets, counts)
    res = root / comp
    kitti.write_labels(root / "val.txt", res / "data", car=files.get("Car"), ped=files.get("Pedestrian"),
                       cyc=files.get("Cyclist"))
    return res


def test_det_file_and_label_formats(tmp_path):
    from mscnn_b200 import kitti
    dets = np.zeros((2, 3, 5), np.float32)
    dets[0, 0] = [10.123456, 20.5, 30.25, 40.0, 0.987654]
    dets[1, 0] = [1234.5678, 0.0, 7.0, 8.0, 1e-5]
    dets[1, 1] = [5.0, 6.0, 7.0, 8.0, 0.5]
    f = tmp_path / "d.txt"
    kitti.write_det_file(f, dets, np.array([1, 2], np.int32))
    assert f.read_text().splitlines() == ["1,10.123,20.5,30.25,40,0.98765", "2,1234.6,0,7,8,1e-05", "2,5,6,7,8,0.5"]
    (tmp_path / "val.txt").write_text("000007\n000123\n")
    kitti.write_labels(tmp_path / "val.txt", tmp_path / "r" / "data", car=f)
    a = (tmp_path / "r" / "data" / "000007.txt").read_text()
    assert a == "Car -1 -1 -10 10.12 20.50 40.37 60.50 -1 -1 -1 -1000 -1000 -1000 -10 987.65 \n"
    b = (tmp_path / "r" / "data" / "000123.txt").read_text().splitlines()
    assert len(b) == 2 and b[1].startswith("Car -1 -1 -10 5.00 6.00 12.00 14.00 ")


def _statistics(res):
    """{path under the result directory: bytes} of every statistics / plot-data file an evaluation wrote."""
    return {str(f.relative_to(res)): f.read_bytes() for f in [*res.glob("stats_*.txt"), *res.glob("plot/*.txt")]}


def _golden_statistics(d):
    return {f.name.replace("plot_", "plot/", 1) if f.name.startswith("plot_") else f.name: f.read_bytes()
            for f in d.glob("*.txt")}


@pytest.mark.parametrize("seed,n", [(7, 24), (11, 40), (3, 5)])
def test_evaluate_byte_identical_to_reference_tool(tmp_path, seed, n):
    """Every file this evaluator writes equals what the reference tool wrote for the same result files; no
    orientation statistics without a valid alpha."""
    from mscnn_b200 import kitti
    ids, rows = make_dataset(tmp_path, n_images=n, seed=seed)
    ours = _write_results(tmp_path, rows, n, "ours")
    ap = kitti.evaluate(tmp_path / "label_2", ours, tmp_path / "val.txt")
    got, want = _statistics(ours), _golden_statistics(GOLDEN / GOLDEN_CASES[seed, n])
    assert sorted(got) == sorted(want)
    for rel in want:
        assert got[rel] == want[rel], rel
    for cls in ("car", "pedestrian", "cyclist"):
        assert not (ours / f"stats_{cls}_orientation.txt").exists()
        tab = np.loadtxt(ours / f"plot/{cls}_detection.txt")
        assert np.allclose(ap[cls], 100 * tab[0:41:4, 1:4].mean(0), atol=1e-4)


def test_evaluate_with_orientation_and_missing_classes(tmp_path):
    """Result files that carry a valid alpha switch the orientation statistics on; classes never detected are
    not evaluated (evaluate_object.cpp:124-134)."""
    from mscnn_b200 import kitti
    ids, rows = make_dataset(tmp_path, n_images=16, seed=21)
    write_oriented_car_results(tmp_path / "ours", ids, rows)
    ap = kitti.evaluate(tmp_path / "label_2", tmp_path / "ours", tmp_path / "val.txt")
    got, want = _statistics(tmp_path / "ours"), _golden_statistics(GOLDEN / "orientation_seed21_n16")
    assert sorted(got) == sorted(want)
    for rel in ("stats_car_detection.txt", "stats_car_orientation.txt", "plot/car_detection.txt", "plot/car_orientation.txt"):
        assert got[rel] == want[rel], rel
    assert ap["pedestrian"] is None and ap["cyclist"] is None and ap["car"] is not None
    assert not (tmp_path / "ours" / "stats_pedestrian_detection.txt").exists()


def test_evaluate_against_committed_reference_output(tmp_path):
    """Same comparison without the reference tool: its output for seed 7 / 24 images is committed."""
    from mscnn_b200 import kitti
    ids, rows = make_dataset(tmp_path, n_images=24, seed=7)
    ours = _write_results(tmp_path, rows, 24, "ours")
    kitti.evaluate(tmp_path / "label_2", ours, tmp_path / "val.txt")
    for f in sorted(GOLDEN.glob("*.txt")):
        rel = f.name.replace("plot_", "plot/") if f.name.startswith("plot_") else f.name
        assert (ours / rel).read_bytes() == f.read_bytes(), rel
    assert len(list(GOLDEN.glob("*.txt"))) == 6


def test_evaluate_perfect_and_empty(tmp_path):
    """Known answers: 80 ground-truth cars (>= 2 per recall step, so all 41 recall points are reached), every one
    detected exactly -> precision 1 everywhere, AP 100; a missing result file is an error, not a crash."""
    from mscnn_b200 import capi, kitti
    gt = tmp_path / "label_2"
    gt.mkdir()
    (tmp_path / "val.txt").write_text("".join(f"{i:06d}\n" for i in range(4)))
    rows = []
    for img in range(4):
        lines = []
        for k in range(20):
            x, y = 10 + 120 * (k % 10), 20 + 150 * (k // 10)
            lines.append(f"Car 0.00 0 1.00 {x:.2f} {y:.2f} {x + 100:.2f} {y + 80:.2f} 1.5 1.6 3.9 1 1.5 20 1.0\n")
            rows.append([img + 1, x, y, 100, 80, 0.5 + 0.005 * (20 * img + k)])
        (gt / f"{img:06d}.txt").write_text("".join(lines))
    dets, counts = rows_to_padded(np.array(rows, dtype=np.float64), 4)
    kitti.write_det_file(tmp_path / "car.txt", dets, counts)
    kitti.write_labels(tmp_path / "val.txt", tmp_path / "res" / "data", car=tmp_path / "car.txt")
    ap = kitti.evaluate(gt, tmp_path / "res", tmp_path / "val.txt")
    assert ap["car"] == (100.0, 100.0, 100.0) and ap["pedestrian"] is None
    with pytest.raises(capi.MscnnError):
        kitti.evaluate(gt, tmp_path / "nowhere", tmp_path / "val.txt")
