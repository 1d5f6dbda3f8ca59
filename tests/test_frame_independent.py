"""pipeline.run_frame_independent (node mode from raw scans) driven by an oracle-backed stand-in of the device handle, without
a GPU: the counter rule that picks the processed nodes, the step sequencing, the final save_static_map.  The stand-in is the
reference's own query preparation (voxelize_preserving_labels + lidar -> body) followed by fetch_VoI + ERASOR per node on the
same initial map, the verdicts ANDed; tests/test_gpu_scans.py checks the device against it bit for bit."""
import ctypes
import os

import numpy as np

from erasor_b200 import kitti, mapgen, pipeline, params as P


def lidar2body_matrix(oracle_mod, l2b):
    """tf_lidar2body_ = geoPose2eigen(pose) * Identity, in float without contraction (OfflineMapUpdater.cpp:89-104)"""
    G = oracle_mod.pose_to_matrix(np.asarray(l2b, dtype=np.float64))
    I = np.eye(4, dtype=np.float32)
    T = np.zeros((4, 4), dtype=np.float32)
    for r in range(4):
        for c in range(4):
            acc = np.float32(0.0)
            for k in range(4):
                acc = np.float32(acc + np.float32(G[r, k] * I[k, c]))
            T[r, c] = acc
    return T


def oracle_query(oracle_mod, scan, leaf, l2b):
    """what callback_node hands to ERASOR::set_inputs (OfflineMapUpdater.cpp:237-241)"""
    return oracle_mod.transform(oracle_mod.voxelize(scan, leaf), lidar2body_matrix(oracle_mod, l2b))


class OracleNodeMode:
    """process_scans / save_static_map of the device handle, restated with the oracle (the frame-independent semantics)."""

    def __init__(self, oracle_mod, up, ep, initial_map):
        self.o = oracle_mod
        self.ep = ep
        self.map = np.ascontiguousarray(initial_map, dtype=np.float32)
        self.keep = np.ones(len(self.map), dtype=np.uint8)
        self.frame_keep, self.stats, self.queries = [], [], []

    def process_scans(self, poses7, scans, offsets, query_voxel_size, lidar2body, voi_max_range):
        er = self.o.Oracle(self.ep)
        for f in range(len(poses7)):
            scan = scans[int(offsets[f]):int(offsets[f + 1])]
            q = oracle_query(self.o, scan, query_voxel_size, lidar2body)
            voi, idx = self.o.fetch_voi(self.map, poses7[f], voi_max_range if voi_max_range > 0 else self.ep.max_range)
            er.run(voi, q)
            _, rej = er.cloud(er.MAP_REJECTED)
            k = np.ones(len(self.map), dtype=np.uint8)
            k[idx[rej]] = 0
            self.keep &= k
            self.frame_keep.append(k)
            self.stats.append((len(voi), len(er.planes()), len(rej)))
            self.queries.append(q)
        er.close()

    def save_static_map(self, voxel_size):
        return self.o.voxelize(self.map[self.keep == 1], voxel_size)

    def close(self):
        pass


def _drive(tmp_path, oracle_mod, n_frames=10):
    from test_pipeline import YAML, _write_drive
    root = _write_drive(tmp_path, n_frames=n_frames)
    cfg = tmp_path / "cfg.yaml"
    cfg.write_text(YAML)
    ep, up = P.load_yaml(str(cfg))
    nodes = list(kitti.iter_nodes(root, "99", 0, n_frames, 1))
    _, naive = mapgen.build_map(nodes, leafsize=float(up.map_voxel_size), voxelize=lambda c, leaf: oracle_mod.voxelize(c, leaf))
    return ep, up, nodes, naive


def test_run_frame_independent_with_oracle_stand_in(oracle_mod, tmp_path):
    ep, up, nodes, naive = _drive(tmp_path, oracle_mod)
    stand_ins = []

    def make(u, e, m):
        stand_ins.append(OracleNodeMode(oracle_mod, u, e, m))
        return stand_ins[-1]

    res = pipeline.run_frame_independent(nodes, naive, up, ep, nodes_per_step=3, make_handle=make, out_dir=str(tmp_path / "out"))
    # the processed nodes are exactly those the reference's callback_node processes
    upd = oracle_mod.OracleUpdater(up, ep, naive)
    processed = [i for i, (seq, odom, cloud) in enumerate(nodes) if upd.callback_node(int(seq), odom, cloud)]
    upd.close()
    assert res["nodes"] == len(nodes) and res["processed_scans"] == len(processed) > 0
    # ... and their verdicts, each against the initial map, ANDed, give the saved map
    keep = np.ones(len(naive), dtype=np.uint8)
    for i in processed:
        _, odom, cloud = nodes[i]
        q = oracle_query(oracle_mod, cloud, float(up.query_voxel_size), up.lidar2body)
        voi, idx = oracle_mod.fetch_voi(naive, odom, float(up.max_range))
        er = oracle_mod.Oracle(ep)
        er.run(voi, q)
        _, rej = er.cloud(er.MAP_REJECTED)
        keep[idx[rej]] = 0
        er.close()
    assert (keep == 0).any()
    expect = oracle_mod.voxelize(naive[keep == 1], float(up.map_voxel_size))
    assert np.array_equal(res["static_map"].view(np.uint32), expect.view(np.uint32))
    assert np.array_equal(stand_ins[0].keep, keep)
    q = res["quality"]
    assert 0.0 <= q["PR"] <= 100.0 and 0.0 < q["RR"] <= 100.0
    assert os.path.exists(tmp_path / "out" / "99_frame_independent_result.pcd")


def test_step_size_does_not_change_the_result(oracle_mod, tmp_path):
    ep, up, nodes, naive = _drive(tmp_path, oracle_mod, n_frames=8)
    make = lambda u, e, m: OracleNodeMode(oracle_mod, u, e, m)
    a = pipeline.run_frame_independent(nodes, naive, up, ep, nodes_per_step=1, make_handle=make)
    b = pipeline.run_frame_independent(nodes, naive, up, ep, nodes_per_step=20, make_handle=make)
    assert np.array_equal(a["static_map"].view(np.uint32), b["static_map"].view(np.uint32))


def test_scan_entry_points_are_exported():
    from erasor_b200 import capi
    L = ctypes.CDLL(capi.LIB_PATH)          # loads without a GPU
    for s in ("erasor_process_scans", "erasor_process_scans_async", "erasor_get_scan_queries", "erasor_save_static_map"):
        assert hasattr(L, s) and s in capi.EXPORTS, s
    assert L.erasor_abi_version() == 2
    assert ctypes.sizeof(capi.ScanParamsC) == 64
