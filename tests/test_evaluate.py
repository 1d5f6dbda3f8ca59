"""CPU suite: the PR/RR port (erasor_b200/evaluate.py) against the reference's own scripts/analysis_runner.py, whose
output on a crop of oracle output is stored in tests/golden/analysis_runner/pr_rr.npz (tests/golden/make_pr_rr_golden.py)."""
import os
import re

import numpy as np
import pytest

from erasor_b200 import evaluate as E
from erasor_b200 import params as P
from erasor_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "analysis_runner", "pr_rr.npz")


@pytest.fixture(scope="module")
def run_pass(oracle_mod):
    sc = synth.Scene(seed=41, length=40.0, n_nodes=17, n_dynamic=6)
    kw = dict(n_beams=24, n_az=480)
    nodes = list(range(17))
    m = sc.build_map(nodes, voxel=0.2, **kw)
    ep, up = P.preset("seq_05"), P.updater_preset("seq_05")
    up.removal_interval = 2
    o = oracle_mod.OracleUpdater(up, ep, m)
    for k in nodes:
        o.callback_node(k, sc.pose7(k), sc.scan(k, seed_offset=3, **kw))
    est = o.save_static_map(0.2)
    return m, est


def test_pr_rr_moves_the_right_way(run_pass):
    gt, est = run_pass
    before = E.evaluate(gt, gt)
    after = E.evaluate(gt, est)
    assert before["PR"] == 100.0 and before["RR"] == 0.0
    assert after["RR"] > 30.0 and after["PR"] > 80.0, after      # the pass erases dynamic trails and keeps most static points


def test_matches_reference_script(tmp_path):
    z = np.load(GOLDEN)
    gp, ep_ = str(tmp_path / "gt.pcd"), str(tmp_path / "est.pcd")
    E.write_pcd_ascii(gp, z["gt"])
    E.write_pcd_ascii(ep_, z["est"])
    mine = E.evaluate(E.read_pcd_ascii(gp), E.read_pcd_ascii(ep_))
    txt = str(z["stdout"])
    # the script prints PR / RR / F1 with 3 decimals in a table; find them
    nums = [float(x) for x in re.findall(r"-?\d+\.\d+", txt)]
    assert any(abs(v - mine["PR"]) < 2e-3 for v in nums), (mine, txt[-800:])
    assert any(abs(v - mine["RR"]) < 2e-3 for v in nums), (mine, txt[-800:])
