"""Generates tests/golden/analysis_runner/pr_rr.npz -- known answer of the upstream ERASOR evaluator for tests/test_evaluate.py.

Two labelled clouds, a crop of an offline pass of the oracle (ground truth = the initial map, estimate = the static map it
saves; the crop keeps dynamic trails and static points next to them) are written as ASCII PCDs with
erasor_b200.evaluate.write_pcd_ascii and handed to ERASOR's own scripts/analysis_runner.py, run unchanged; its stdout is
stored beside the clouds.  Run from the repo root:
    python tests/golden/make_pr_rr_golden.py <ERASOR checkout>/scripts/analysis_runner.py
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from erasor_b200 import evaluate as E  # noqa: E402
from erasor_b200 import params as P  # noqa: E402
from erasor_b200 import synth  # noqa: E402
from oracle import oracle_py as O  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
BOX = (10.0, 25.0, -4.0, 4.0)       # x0 x1 y0 y1, metres


def main(runner):
    sc = synth.Scene(seed=41, length=40.0, n_nodes=17, n_dynamic=6)
    kw = dict(n_beams=24, n_az=480)
    nodes = list(range(17))
    m = sc.build_map(nodes, voxel=0.2, **kw)
    ep, up = P.preset("seq_05"), P.updater_preset("seq_05")
    up.removal_interval = 2
    o = O.OracleUpdater(up, ep, m)
    for k in nodes:
        o.callback_node(k, sc.pose7(k), sc.scan(k, seed_offset=3, **kw))
    est = o.save_static_map(0.2)
    crop = lambda a: np.ascontiguousarray(a[(a[:, 0] >= BOX[0]) & (a[:, 0] < BOX[1]) & (a[:, 1] >= BOX[2]) & (a[:, 1] < BOX[3])])
    gt, est = crop(m), crop(est)
    with tempfile.TemporaryDirectory() as d:
        E.write_pcd_ascii(os.path.join(d, "gt.pcd"), gt)
        E.write_pcd_ascii(os.path.join(d, "est.pcd"), est)
        out = subprocess.run([sys.executable, os.path.abspath(runner), "--gt", "gt.pcd", "--est", "est.pcd"], cwd=d,
                             capture_output=True, text=True, check=True)
    np.savez_compressed(os.path.join(HERE, "analysis_runner", "pr_rr.npz"), gt=gt, est=est, stdout=np.str_(out.stdout))
    print(len(gt), len(est))
    print(out.stdout)


if __name__ == "__main__":
    main(sys.argv[1])
