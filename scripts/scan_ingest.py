"""scan_ingest.py -- node mode from raw LiDAR scans (erasor_process_scans) on the seq-05 twin, against the same step fed
prepared queries (erasor_process_nodes, bench.py's headline path).

The workload is bench.py's: the seq-05 synthetic twin, 20 processed nodes per step, four handles (lanes) fed round-robin with
asynchronous submissions against one resident map.  Raw scans are synth.Scene.scan of the same nodes (LiDAR frame,
lidar2body = (0, 0, 1.73, 0, 0, 0, 1)).  Arms, one JSON line each:
  (a) raw x y z i scans from pinned host memory      (b) raw packed x y z scans from pinned host memory
  (c) raw scans already resident in HBM              (d) process_nodes with prepared queries resident in HBM (reference point)
Each arm: median of three timed blocks of --steps steps (wall clock between two device synchronisations).  A last line
records the host preparation the raw-scan path replaces (oracle voxelise + lidar -> body, one core, per scan), the bytes
crossing PCIe per step, the card and its power limit, and the frame-independent PR/RR with raw-scan queries beside the
sequential updater's on the same nodes.

    python scripts/scan_ingest.py [--steps 30] [--out profiles/r03/scan_ingest.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2B = [0.0, 0.0, 1.73, 0.0, 0.0, 0.0, 1.0]


def workload(frames):
    from erasor_b200 import synth
    cache = os.path.join(tempfile.gettempdir(), f"erasor_b200_scan_ingest_f{frames}.npz")
    if os.path.exists(cache):
        z = np.load(cache)
        return {k: z[k] for k in z.files}
    w = synth.make_frames(seed=5, n_frames=frames, preset_max_range=60.0, n_map_nodes=161, n_beams=64, n_az=1800, length=160.0,
                          n_dynamic=12, query_voxel=0.2, map_stride=2)
    ks = [f[2] for f in w["frames"]]
    d = dict(map_world=w["map_world"], poses=np.stack([w["scene"].pose7(k) for k in ks]), nodes=np.array(ks))
    for i, f in enumerate(w["frames"]):
        d[f"q_{i}"] = f[1]
        d[f"s_{i}"] = w["scene"].scan(f[2], seed_offset=17)
    np.savez(cache, **d)
    return d


def power_limit_w():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--lanes", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from erasor_b200 import capi, params, pipeline, evaluate
    from oracle import oracle_py
    oracle_py.build()

    d = workload(args.frames)
    F = args.frames
    p = params.preset("seq_05").replace(skip_voxelize=1)
    map_world = d["map_world"]
    poses = np.ascontiguousarray(d["poses"], dtype=np.float64)
    scans = [d[f"s_{i}"] for i in range(F)]
    qs = [d[f"q_{i}"] for i in range(F)]
    so = np.cumsum([0] + [len(s) for s in scans]).astype(np.uint64)
    qo = np.cumsum([0] + [len(q) for q in qs]).astype(np.uint64)
    S = np.ascontiguousarray(np.concatenate(scans), dtype=np.float32)
    Q = np.ascontiguousarray(np.concatenate(qs), dtype=np.float32)
    dev = torch.device("cuda", 0)
    gmap = capi.Map(map_world)
    lanes = [capi.Handle(p) for _ in range(args.lanes)]
    for h in lanes:
        h.attach_map(gmap)
    sp = capi.scan_params(0.2, L2B)
    hS = torch.from_numpy(S).pin_memory()
    hS3 = torch.from_numpy(np.ascontiguousarray(S[:, :3])).pin_memory()
    dS = [torch.from_numpy(S).to(dev) for _ in range(2)]
    dQ = [torch.from_numpy(Q).to(dev) for _ in range(2)]
    torch.cuda.synchronize()

    arms = {
        "a_raw_xyzi_pinned_host": lambda i, h: h.process_scans_ptr(sp, poses, hS.data_ptr(), so, 0.0, 0, 0, capi.PTR_HOST, asynchronous=True),
        "b_raw_xyz_pinned_host": lambda i, h: h.process_scans_ptr(sp, poses, hS3.data_ptr(), so, 0.0, 0, 0, capi.PTR_HOST | capi.PTR_QUERY_XYZ, asynchronous=True),
        "c_raw_xyzi_resident": lambda i, h: h.process_scans_ptr(sp, poses, dS[i % 2].data_ptr(), so, 0.0, 0, 0, capi.PTR_DEVICE, asynchronous=True),
        "d_prepared_queries_resident": lambda i, h: h.process_nodes_ptr(poses, dQ[i % 2].data_ptr(), qo, 0.0, 0, 0, capi.PTR_DEVICE, asynchronous=True),
    }
    bytes_step = {"a_raw_xyzi_pinned_host": 16 * int(so[-1]), "b_raw_xyz_pinned_host": 12 * int(so[-1]), "c_raw_xyzi_resident": 0,
                  "d_prepared_queries_resident": 0}
    name = torch.cuda.get_device_name(0)
    plim = power_limit_w()
    lines = []
    for arm, submit in arms.items():
        L = len(lanes)
        for i in range(2 * L):                                   # warm: every (lane, buffer) pair captured once
            lanes[i % L].wait()
            submit(i, lanes[i % L])
        for h in lanes:
            h.wait()
        blocks = []
        for rep in range(3):
            gmap.reset_keep()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(args.steps):
                lanes[i % L].wait()
                submit(i, lanes[i % L])
            for h in lanes:
                h.wait()
            torch.cuda.synchronize()
            blocks.append(1000 * (time.perf_counter() - t0))
        ms = float(np.median(blocks))
        rec = {"arm": arm, "scans_per_s": round(args.steps * F / (ms / 1000), 1), "ms_per_step": round(ms / args.steps, 4),
               "blocks_ms": [round(b, 3) for b in blocks], "steps": args.steps, "nodes_per_step": F, "lanes": L,
               "pcie_h2d_bytes_per_step": bytes_step[arm], "scan_points_per_step": int(so[-1]), "query_points_per_step": int(qo[-1]),
               "gpu": name, "power_limit_w": plim}
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    # host preparation this path replaces: oracle voxelise + lidar -> body, one core
    T = oracle_py.pose_to_matrix(np.array(L2B))
    t0 = time.perf_counter()
    for s in scans:
        oracle_py.transform(oracle_py.voxelize(s, 0.2), T)
    host_ms = 1000 * (time.perf_counter() - t0) / F

    # quality: frame-independent mode with raw-scan queries vs the sequential updater on the same nodes
    ep = params.preset("seq_05")
    up = params.updater_preset("seq_05")
    from erasor_b200 import synth
    scene = synth.Scene(seed=5, length=160.0, n_nodes=161, n_dynamic=12)
    nodes = []                                                   # bench.py's offline pass: 161 nodes, every 8th processed
    for k in range(161):
        proc = (k + 1) % up.removal_interval == 0
        nodes.append((k, scene.pose7(k), scene.scan(k, seed_offset=17) if proc else np.zeros((0, 4), np.float32)))
    fi = pipeline.run_frame_independent(nodes, map_world, up, ep, nodes_per_step=F)
    seq = pipeline.run_offline(nodes, map_world, up, ep)
    seq_q = evaluate.evaluate(map_world, seq["static_map"], voxelsize=0.2)
    rec = {"arm": "context", "host_prep_ms_per_scan_one_core": round(host_ms, 3), "host_prep": "oracle voxelize_preserving_labels + transform, 0.2 m",
           "pcie_bytes_per_step": {k: v for k, v in bytes_step.items()}, "gpu": name, "power_limit_w": plim,
           "frame_independent_raw_scans": {"processed": fi["processed_scans"], "PR": round(fi["quality"]["PR"], 3), "RR": round(fi["quality"]["RR"], 3),
                                           "static_map_points": int(len(fi["static_map"]))},
           "sequential_updater": {"processed": seq["processed_scans"], "PR": round(seq_q["PR"], 3), "RR": round(seq_q["RR"], 3),
                                  "static_map_points": int(len(seq["static_map"]))}}
    lines.append(rec)
    print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in lines:
                fh.write(json.dumps(r) + "\n")
    for h in lanes:
        h.close()
    gmap.close()


if __name__ == "__main__":
    main()
