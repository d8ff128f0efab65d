"""Seeded synthetic KITTI-style ground truth and detection lists for the evaluator tests (tests/test_kitti_eval.py,
tests/golden/make_kitti_golden.py).  Not a dataset: random boxes with the label fields the evaluation reads."""
from pathlib import Path

import numpy as np

GT_TYPES = ["Car", "Car", "Car", "Van", "Truck", "Pedestrian", "Pedestrian", "Person_sitting", "Cyclist", "Tram", "Misc",
            "DontCare"]


def make_dataset(root: Path, n_images: int = 24, seed: int = 7, with_alpha: bool = False):
    """Writes root/label_2/<id>.txt, root/val.txt and returns per-class detection rows [img x y w h score]
    (img = 1-based list position) in the layout run_mscnn_detection.m saves."""
    rng = np.random.default_rng(seed)
    gt_dir = root / "label_2"
    gt_dir.mkdir(parents=True, exist_ok=True)
    ids = sorted(rng.choice(7481, size=n_images, replace=False).tolist())
    (root / "val.txt").write_text("".join(f"{i:06d}\n" for i in ids))
    dets = {"Car": [], "Pedestrian": [], "Cyclist": []}
    for pos, img in enumerate(ids, start=1):
        lines = []
        for _ in range(int(rng.integers(0, 9))):
            t = GT_TYPES[int(rng.integers(len(GT_TYPES)))]
            w, h = float(rng.uniform(15, 260)), float(rng.uniform(12, 160))
            x1, y1 = float(rng.uniform(0, 1242 - w)), float(rng.uniform(0, 375 - h))
            if t == "DontCare":
                trunc, occ, alpha = -1.0, -1, -10.0
            else:
                trunc = float(rng.choice([0.0, 0.0, 0.1, 0.2, 0.4, 0.7]))
                occ = int(rng.choice([0, 0, 1, 2, 3]))
                alpha = float(rng.uniform(-3.1, 3.1))
            lines.append(f"{t} {trunc:.2f} {occ} {alpha:.2f} {x1:.2f} {y1:.2f} {x1 + w:.2f} {y1 + h:.2f} "
                         f"1.50 1.60 3.90 1.00 1.50 20.00 {alpha:.2f}")
            if t in dets and rng.random() < 0.85:          # a detection near this object, sometimes too loose
                j = rng.normal(0, 0.06 if rng.random() < 0.7 else 0.25, size=4)
                dets[t].append([pos, x1 + j[0] * w, y1 + j[1] * h, w * (1 + j[2]), h * (1 + j[3]), float(rng.uniform(0.2, 1.0))])
                if rng.random() < 0.2:                      # a duplicate with a lower score
                    dets[t].append([pos, x1 + 2, y1 + 1, w, h, float(rng.uniform(0.05, 0.5))])
            elif t in ("Van", "DontCare", "Person_sitting") and rng.random() < 0.6:
                cls = "Car" if t != "Person_sitting" else "Pedestrian"
                dets[cls].append([pos, x1 + 1, y1 + 1, w - 2, h - 2, float(rng.uniform(0.1, 0.9))])
        (gt_dir / f"{img:06d}.txt").write_text("".join(l + "\n" for l in lines))
        for cls in dets:                                     # false positives
            for _ in range(int(rng.integers(0, 3))):
                w, h = float(rng.uniform(20, 200)), float(rng.uniform(20, 120))
                dets[cls].append([pos, float(rng.uniform(0, 1242 - w)), float(rng.uniform(0, 375 - h)), w, h,
                                  float(rng.uniform(0.0, 0.7))])
    return ids, {k: np.asarray(v, dtype=np.float64).reshape(-1, 6) for k, v in dets.items()}


def write_oriented_car_results(res: Path, ids, rows) -> None:
    """KITTI result files under res/data carrying a valid alpha per Car row (switches the orientation statistics on);
    no Pedestrian / Cyclist rows."""
    rng = np.random.default_rng(0)
    (res / "data").mkdir(parents=True)
    for pos, img in enumerate(ids, start=1):
        lines = []
        for x in rows["Car"][rows["Car"][:, 0] == pos]:
            lines.append(f"Car -1 -1 {rng.uniform(-3, 3):.2f} {x[1]:.2f} {x[2]:.2f} {x[1] + x[3]:.2f} {x[2] + x[4]:.2f} "
                         f"-1 -1 -1 -1000 -1000 -1000 -10 {x[5] * 1000:.2f} \n")
        (res / "data" / f"{img:06d}.txt").write_text("".join(lines))


def rows_to_padded(rows: np.ndarray, n_images: int):
    """[img x y w h score] rows -> (dets [N][max][5] float32, counts [N]) as Net.detect returns them."""
    counts = np.array([(rows[:, 0] == i + 1).sum() for i in range(n_images)], dtype=np.int32)
    dets = np.zeros((n_images, max(int(counts.max()), 1), 5), dtype=np.float32)
    for i in range(n_images):
        sel = rows[rows[:, 0] == i + 1][:, 1:]
        dets[i, : len(sel)] = sel
    return dets, counts
