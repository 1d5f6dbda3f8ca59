"""Preservation Rate / Rejection Rate / F1 exactly as the reference's evaluator defines them
(reference scripts/analysis.py:124-155,189-191; identical in scripts/analysis_runner.py:74-105):
1-NN from every ground-truth point into the estimate, inlier if the distance is below voxelsize*sqrt(3)/2;
PR = GT-static inliers whose match is static / GT static; RR = (GT dynamic - GT-dynamic inliers whose match is
dynamic) / GT dynamic; dynamic = SemanticKITTI classes 252..259 carried numerically in `intensity`.
Host-side quality judge, not part of the path.  tests/test_evaluate.py checks it against the stored output of the
reference's own script (tests/golden/analysis_runner/pr_rr.npz).
"""
from __future__ import annotations

import numpy as np

DYNAMIC_CLASSES = (252, 253, 254, 255, 256, 257, 258, 259)


def semantic(intensity: np.ndarray) -> np.ndarray:
    return intensity.astype(np.uint32) & 0xFFFF


def evaluate(gt_xyzi: np.ndarray, est_xyzi: np.ndarray, voxelsize: float = 0.2) -> dict:
    from sklearn.neighbors import NearestNeighbors
    gt_xyz, est_xyz = gt_xyzi[:, :3].astype(np.float32), est_xyzi[:, :3].astype(np.float32)
    gt_sem, est_sem = semantic(gt_xyzi[:, 3]), semantic(est_xyzi[:, 3])
    gt_dyn_all = np.isin(gt_sem, DYNAMIC_CLASSES)
    ns_gt, nd_gt = int((~gt_dyn_all).sum()), int(gt_dyn_all.sum())
    nn = NearestNeighbors(n_neighbors=1, algorithm="kd_tree").fit(est_xyz)
    dists, idx = nn.kneighbors(gt_xyz)
    dists, idx = dists.reshape(-1), idx.reshape(-1)
    is_in = dists < voxelsize * np.sqrt(3) / 2
    gt_is_dyn = np.isin(gt_sem[is_in], DYNAMIC_CLASSES)
    est_is_dyn = np.isin(est_sem[idx[is_in]], DYNAMIC_CLASSES)
    preserved_static = int(np.sum((~gt_is_dyn) & (~est_is_dyn)))
    preserved_dynamic = int(np.sum(gt_is_dyn & est_is_dyn))
    pr = preserved_static / ns_gt * 100.0 if ns_gt else 0.0
    rr = (nd_gt - preserved_dynamic) / nd_gt * 100.0 if nd_gt else 0.0
    f1 = 2 * (pr / 100) * (rr / 100) / ((pr / 100) + (rr / 100)) if (pr + rr) > 0 else 0.0
    return {"gt_static": ns_gt, "gt_dynamic": nd_gt, "preserved_static": preserved_static,
            "preserved_dynamic": preserved_dynamic, "PR": pr, "RR": rr, "F1": f1}


def write_pcd_ascii(path: str, xyzi: np.ndarray):
    """ASCII PCD in the layout pcl::io::savePCDFileASCII produces for PointXYZI (what analysis_runner.py reads)."""
    n = len(xyzi)
    with open(path, "w") as f:
        f.write("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z intensity\nSIZE 4 4 4 4\nTYPE F F F F\n"
                f"COUNT 1 1 1 1\nWIDTH {n}\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS {n}\nDATA ascii\n")
        np.savetxt(f, xyzi, fmt="%.8g")


def read_pcd_ascii(path: str) -> np.ndarray:
    with open(path, "r") as f:
        fields, n = None, None
        for line in f:
            line = line.strip()
            if line.startswith("FIELDS"):
                fields = line.split()[1:]
            elif line.startswith("POINTS"):
                n = int(line.split()[1])
            elif line.startswith("DATA"):
                assert line.split()[1] == "ascii"
                break
        arr = np.loadtxt(f, dtype=np.float64, max_rows=n).reshape(-1, len(fields))
    cols = {name: arr[:, i] for i, name in enumerate(fields)}
    return np.stack([cols["x"], cols["y"], cols["z"], cols["intensity"]], axis=1).astype(np.float32)
