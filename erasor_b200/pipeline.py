"""The reference's three-stage workflow in one call, ROS stripped (README "How to run": mapgen -> offline_map_updater ->
scripts/analysis_runner.py):

    nodes (erasor_b200.kitti.iter_nodes, or any iterable of (seq, odom7, cloud))
      -> naive map            erasor_b200.mapgen           (src/mapgen)
      -> static map           capi.Updater, one erasor_updater_process_node per node + save_static_map
                              (OfflineMapUpdater::callback_node / save_static_map, OfflineMapUpdater.cpp:174-330)
      -> PR / RR              erasor_b200.evaluate         (scripts/analysis_runner.py)

Everything heavy runs on the device behind the C ABI; this module only sequences the calls.  The updater and the voxeliser are
injectable so that tests/test_pipeline.py can drive the same code with the oracle's objects on a machine without a GPU.
"""
from __future__ import annotations

import os
from typing import Callable, Iterable, Optional, Tuple

import numpy as np

from . import evaluate, kitti, mapgen, params

Node = Tuple[int, np.ndarray, np.ndarray]


def run_offline(nodes: Iterable[Node], initial_map: np.ndarray, up, ep, make_updater: Optional[Callable] = None,
                save_voxel_size: Optional[float] = None) -> dict:
    """Feed every node to the map updater, then save_static_map.  make_updater(up, ep, initial_map) must return an object with
    process_node(seq, odom7, cloud) -> bool, save_static_map(voxel) -> cloud (capi.Updater by default: needs a CUDA device)."""
    if make_updater is None:
        from . import capi
        make_updater = lambda u, e, m: capi.Updater(u, e, m)
    upd = make_updater(up, ep, np.ascontiguousarray(initial_map, dtype=np.float32))
    seen = processed = 0
    for seq, odom, cloud in nodes:
        seen += 1
        processed += 1 if upd.process_node(int(seq), odom, cloud) else 0
    static_map = upd.save_static_map(up.map_voxel_size if save_voxel_size is None else save_voxel_size)
    if hasattr(upd, "close"):
        upd.close()
    return {"static_map": static_map, "nodes": seen, "processed_scans": processed}


def run_sequence(nodes, up, ep, voxelize: Optional[mapgen.Voxelizer] = None, make_updater: Optional[Callable] = None,
                 map_leafsize: Optional[float] = None, out_dir: Optional[str] = None) -> dict:
    """mapgen -> updater -> evaluation on one node list.  GT for PR/RR = the naive map itself (it carries the labels), which is
    how the reference scores a run (analysis_runner.py compares <seq>_..._original / voxelised map with the result)."""
    nodes = list(nodes)
    leaf = float(up.map_voxel_size if map_leafsize is None else map_leafsize)
    original, naive = mapgen.build_map(nodes, leafsize=leaf, is_large_scale=bool(up.is_large_scale), voxelize=voxelize)
    res = run_offline(nodes, naive, up, ep, make_updater=make_updater)
    res["naive_map"] = naive
    res["quality"] = evaluate.evaluate(naive, res["static_map"], voxelsize=0.2)
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        name = getattr(up, "data_name", "seq")
        evaluate.write_pcd_ascii(os.path.join(out_dir, f"{name}_naive_map.pcd"), naive)
        evaluate.write_pcd_ascii(os.path.join(out_dir, f"{name}_result.pcd"), res["static_map"])      # save_static_map's file name (:193)
    return res


class _DeviceNodeMode:
    """The resident map plus one handle attached to it: the default back end of run_frame_independent."""

    def __init__(self, up, ep, initial_map, device: int = 0):
        from . import capi
        self.map = capi.Map(initial_map, device=device)
        self.h = capi.Handle(ep, device=device)
        self.h.attach_map(self.map)

    def process_scans(self, poses7, scans, offsets, query_voxel_size, lidar2body, voi_max_range):
        self.h.process_scans(poses7, scans, offsets, query_voxel_size, lidar2body, voi_max_range=voi_max_range)

    def save_static_map(self, voxel_size: float) -> np.ndarray:
        return self.h.save_static_map(voxel_size)

    def close(self):
        self.h.close()
        self.map.close()


def run_frame_independent(nodes: Iterable[Node], initial_map: np.ndarray, up, ep, nodes_per_step: int = 20, device: int = 0,
                          out_dir: Optional[str] = None, make_handle: Optional[Callable] = None) -> dict:
    """The frame-independent mode from raw scans: every processed node is tested against the same initial map and the verdicts
    are ANDed (DESIGN section 7), instead of the sequential updater's map that changes node by node.  A node is processed by
    the updater's counter rule (call k, 0-based, iff (k + 1) % removal_interval == 0).  Processed nodes go in steps of
    nodes_per_step through erasor_process_scans (voxelise + lidar -> body on the device), then save_static_map at
    up.map_voxel_size.  make_handle(up, ep, initial_map) must return an object with process_scans(poses7, scans, offsets,
    query_voxel_size, lidar2body, voi_max_range), save_static_map(voxel) and close() (default: the device map + handle)."""
    if make_handle is None:
        make_handle = lambda u, e, m: _DeviceNodeMode(u, e, m, device=device)
    initial_map = np.ascontiguousarray(initial_map, dtype=np.float32)
    h = make_handle(up, ep, initial_map)
    step = max(1, int(nodes_per_step))
    seen = processed = 0
    poses, scans = [], []

    def flush():
        if not scans:
            return
        off = np.cumsum([0] + [len(c) for c in scans]).astype(np.uint64)
        cat = np.concatenate(scans) if int(off[-1]) else np.zeros((0, 4), dtype=np.float32)
        h.process_scans(np.stack(poses).astype(np.float64), cat, off, float(up.query_voxel_size), list(up.lidar2body), float(up.max_range))
        poses.clear()
        scans.clear()

    try:
        for seq, odom, cloud in nodes:
            seen += 1
            if seen % int(up.removal_interval) != 0:
                continue
            processed += 1
            poses.append(np.asarray(odom, dtype=np.float64).reshape(7))
            scans.append(np.ascontiguousarray(cloud, dtype=np.float32).reshape(-1, 4))
            if len(scans) == step:
                flush()
        flush()
        static_map = h.save_static_map(float(up.map_voxel_size))
    finally:
        if hasattr(h, "close"):
            h.close()
    res = {"static_map": static_map, "nodes": seen, "processed_scans": processed, "naive_map": initial_map,
           "quality": evaluate.evaluate(initial_map, static_map, voxelsize=0.2)}
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        name = getattr(up, "data_name", "seq")
        evaluate.write_pcd_ascii(os.path.join(out_dir, f"{name}_frame_independent_result.pcd"), static_map)
    return res


def run_semantickitti(dataset_root: str, sequence: str, init_stamp: int, end_stamp: int, interval: int, config_yaml: str,
                      out_dir: Optional[str] = None, **kw) -> dict:
    """SemanticKITTI files + a reference config/*.yaml -> static map and PR/RR."""
    ep, up = params.load_yaml(config_yaml)
    return run_sequence(kitti.iter_nodes(dataset_root, sequence, init_stamp, end_stamp, interval), up, ep, out_dir=out_dir, **kw)
