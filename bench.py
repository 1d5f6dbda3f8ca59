#!/usr/bin/env python
"""bench.py -- LiDAR scans/sec through R-POD + SRT + R-GPF on the synthetic twin of KITTI seq 05.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (N>1: launched under torch.distributed.run,
one rank per GPU).  One JSON line on rank 0.

Workload (BASELINE.json configs[1]): KITTI seq 05, frames 2350-2670, reference config/seq_05.yaml
(15 rings x 60 sectors @ 60 m, version 3).  161 nodes, every 8th processed (removal_interval 8) = 20 hot-path
frames per offline pass.  No KITTI data exists here, so the twin is a seeded synthetic street scene
(erasor_b200/synth.py): HDL-64-like ray-cast scans, a 0.2 m voxelised accumulated map with moving-object trails.
A "step" = one pass of the hot path over one rank's 20 nodes in the frame-independent mode north_star shards across
GPUs: the global map is uploaded once (OfflineMapUpdater::load_global_map) and stays in HBM; per node the library
gets the pose and the voxelised body-frame query (what callback_node hands to ERASOR::set_inputs) and does
fetch_VoI + R-POD + SRT + R-GPF on the device (erasor_process_nodes).  Weak scaling: every rank gets its own 20 nodes.

value : scans/s, queries already resident in HBM (device pointers), `--lanes` handles fed round-robin with
        asynchronous submissions (consecutive batches overlap on the GPU).
e2e   : scans/s through the same C-ABI call with pinned HOST buffers: poses + queries H2D and the folded keep
        mask of the map D2H inside the timed region, every step.
roofline : the kernel with the largest CUDA-event time per step against the measured HBM peak, plus every kernel's own
        line (`by_kernel`; K1 is the one that moves the path's bytes, R-GPF the latency-bound one).
cpu_baseline : the oracle port (oracle/, restated reference path: fetch_VoI + ERASOR) on one host core, bounded sample.
--impl reference : the same oracle port over all host cores (independent nodes in a process pool).
--config NAME : other BASELINE.json configs (dense twin, 50 M-point VoI, 40x360 x 256 k-point scans); their lines are
        committed under profiles/r02/.  The driver's default stays on seq 05.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FRAMES_PER_PASS = 20          # 161 nodes / removal_interval 8 (config/seq_05.yaml)
N_QUERY_COPIES = 20           # resident arm: rotating query copies, 20 x 6.6 MB > 126 MB L2
CACHE_DIR = os.environ.get("ERASOR_B200_CACHE", "/tmp/erasor_b200_cache")

CONFIGS = {
    # name: (erasor preset, synth kwargs, description)
    "seq05": dict(preset="seq_05", synth=dict(seed=5, n_map_nodes=161, n_beams=64, n_az=1800, length=160.0, n_dynamic=12, query_voxel=0.2, map_stride=2),
                  what="KITTI seq 05 (2350-2670) synthetic twin, config/seq_05.yaml"),
    # SURVEY 8's size estimate for the real sequence (N_m 0.5-1 M, N_q ~40 k): every node in the map, 0.1 deg azimuth steps
    "dense": dict(preset="seq_05", synth=dict(seed=5, n_map_nodes=161, n_beams=64, n_az=3600, length=160.0, n_dynamic=12, query_voxel=0.2, map_stride=1),
                  what="seq 05 twin at the size SURVEY section 8 estimates for the real data (denser scans, every node mapped)"),
    "synthetic40x360": dict(preset="synthetic_40x360", synth=None,
                            what="BASELINE config 5: 262144-point scans, 40 rings x 360 sectors, N_map 2 M shared static map + per-frame pose"),
}


def _cache(path_key, build):
    os.makedirs(CACHE_DIR, exist_ok=True)
    path = os.path.join(CACHE_DIR, path_key)
    if os.path.exists(path):
        z = np.load(path)
        return {k: z[k] for k in z.files}
    d = build()
    tmp = path + f".tmp{os.getpid()}.npz"
    np.savez(tmp, **d)
    os.replace(tmp, path)
    return d


def synth_40x360(total_frames: int):
    """BASELINE config 5.  The reference has no such yaml (nearest: large_scale_05.yaml geometry); N_map is ours to state:
    2 M points in a 240 m x 240 m world -- flat-ish ground (85 %), boxes (static 10 %), moving-object trails (5 %, labels 252);
    each frame = a pose on a circle + a 262144-point scan of the same world without the trails, cropped at 80 m."""
    rng = np.random.default_rng(5)
    n_map, n_q = 2_000_000, 262_144
    def world(n, with_trails):
        xy = rng.uniform(-120.0, 120.0, (n, 2))
        z = 0.05 * np.sin(0.07 * xy[:, 0]) + 0.04 * np.cos(0.05 * xy[:, 1]) + rng.normal(0, 0.02, n) - 1.0
        lab = np.full(n, 40.0)
        k = rng.uniform(size=n)
        box = k < 0.10
        z[box] += rng.uniform(0.2, 2.5, int(box.sum())); lab[box] = 50.0
        if with_trails:
            tr = (k >= 0.10) & (k < 0.15)
            cx = np.round(xy[tr] / 24.0) * 24.0 + 5.0                       # trails: 4 m x 2 m blobs on a 24 m lattice
            xy[tr] = cx + rng.uniform(-1.0, 1.0, (int(tr.sum()), 2)) * np.array([2.0, 1.0])
            z[tr] = -1.0 + rng.uniform(0.1, 1.6, int(tr.sum())); lab[tr] = 252.0
        return np.concatenate([xy, z[:, None], lab[:, None]], axis=1).astype(np.float32)
    map_world = world(n_map, True)
    poses = np.zeros((total_frames, 7))
    qs = []
    for f in range(total_frames):
        a = 2 * np.pi * f / max(total_frames, 1)
        poses[f] = [30.0 * np.cos(a), 30.0 * np.sin(a), 0.0, 0.0, 0.0, np.sin(a / 2), np.cos(a / 2)]
    base = world(3 * n_q, False)                                            # one dense static world, re-cropped per pose
    from erasor_b200 import synth
    for f in range(total_frames):
        T = np.linalg.inv(synth.pose_matrix(poses[f]))
        d2 = (base[:, 0] - poses[f, 0]) ** 2 + (base[:, 1] - poses[f, 1]) ** 2
        sel = base[d2 < 80.0 ** 2]
        sel = sel[rng.choice(len(sel), n_q, replace=len(sel) < n_q)]
        q = sel.copy()
        q[:, :3] = (sel[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
        qs.append(q)
    return map_world, poses, qs


def load_workload(config: str, rank: int, world: int, frames_per_rank: int):
    """One map + world*frames_per_rank nodes along the trajectory (pose + voxelised body-frame query); this rank's share."""
    from erasor_b200 import params, synth
    cfg = CONFIGS[config]
    p = params.preset(cfg["preset"]).replace(skip_voxelize=1)
    total = world * frames_per_rank
    if cfg["synth"] is None:
        def build():
            m, poses, qs = synth_40x360(total)
            return dict(map_world=m, poses=poses, **{f"q_{i}": q for i, q in enumerate(qs)})
        d = _cache(f"{config}_f{total}_v2.npz", build)
    else:
        kw = cfg["synth"]
        def build():
            w = synth.make_frames(n_frames=total, preset_max_range=p.max_range, **kw)
            poses = np.stack([w["scene"].pose7(f[2]) for f in w["frames"]])
            return dict(map_world=w["map_world"], poses=poses, **{f"q_{i}": f[1] for i, f in enumerate(w["frames"])})
        d = _cache(f"{config}_seed{kw['seed']}_n{kw['n_map_nodes']}_s{kw['map_stride']}_az{kw['n_az']}_f{total}_v2.npz", build)
    # strided shard (SURVEY 8e: "contiguous or strided frame ranges per rank"): rank r takes nodes r, r + world, r + 2 world, ...
    # so every rank sees the whole trajectory and the ranks' steps cost about the same (max-over-ranks timing)
    mine = list(range(rank, total, world))
    qs = [d[f"q_{i}"] for i in mine]
    poses = np.ascontiguousarray(d["poses"][mine], dtype=np.float64)
    return p, d["map_world"], poses, qs


def offline_pass_block(p, map_world, device_index):
    """Sequential offline pass through the device-resident OfflineMapUpdater (SURVEY 8f rows 1-3): 161 nodes, every 8th
    processed (config/seq_05.yaml removal_interval 8), raw scans from pinned host memory, map state in HBM.  Wall clock
    around erasor_updater_process_node (it synchronises its stream).  Same pass on the oracle's restated caller loop on
    one host core.  Informational: the driver's headline numbers are `value` / `e2e` above."""
    import torch
    from erasor_b200 import capi, params, synth
    from oracle import oracle_py
    up = params.updater_preset("seq_05")
    ep = params.preset("seq_05")                     # version 3 with in-bin voxelisation, as shipped
    scene = synth.Scene(seed=5, length=160.0, n_nodes=161, n_dynamic=12)
    nodes = list(range(161))
    processed = [k for k in nodes if (k + 1) % up.removal_interval == 0]
    d = _cache("seq05_twin_seed5_scans_ri8.npz", lambda: {f"s_{k}": scene.scan(k, seed_offset=17) for k in processed})
    scans = {k: d[f"s_{k}"] for k in processed}
    empty = np.zeros((0, 4), dtype=np.float32)
    pinned = {k: torch.from_numpy(v).pin_memory() for k, v in scans.items()}
    poses = [scene.pose7(k) for k in nodes]
    best = None
    pass_ms = []
    u = capi.Updater(up, ep, map_world, device=device_index)
    first_map = None
    for rep in range(5):
        if rep:
            u.reset(map_world)                       # load_global_map again; device buffers are kept
        l0 = u.kernel_launch_count()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        nxt = {a: b for a, b in zip(processed, processed[1:])}       # the node processed after each processed node
        u.prefetch_scan_ptr(pinned[processed[0]].data_ptr(), len(scans[processed[0]]), capi.PTR_HOST)
        for k in nodes:
            if k in pinned:
                if k in nxt:                           # look-ahead: the next processed node's scan uploads + voxelises under this node's path
                    u.prefetch_scan_ptr(pinned[nxt[k]].data_ptr(), len(scans[nxt[k]]), capi.PTR_HOST)
                u.process_node_ptr(k, poses[k], pinned[k].data_ptr(), len(scans[k]), capi.PTR_HOST)
            else:
                u.process_node_ptr(k, poses[k], 0, 0, capi.PTR_HOST)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        launches = u.kernel_launch_count() - l0
        n_final = u.map_size()
        pass_ms.append(round(1000 * dt, 2))
        if best is None or dt < best[0]:
            best = (dt, launches, n_final)
        if rep == 0:
            first_map = u.cloud(u.MAP_ARRANGED)
    u.close()
    o = oracle_py.OracleUpdater(up, ep, map_world)
    t0 = time.perf_counter()
    hot = 0.0
    for k in nodes:
        if o.callback_node(k, poses[k], scans.get(k, empty)):
            hot += o.erasor_seconds()
    cpu_dt = time.perf_counter() - t0
    ref_map, _ = o.cloud(o.MAP_ARRANGED)
    same = bool(first_map.shape == ref_map.shape and np.array_equal(first_map.view(np.uint32), ref_map.view(np.uint32)))
    from erasor_b200 import evaluate
    pr = evaluate.evaluate(map_world, first_map)
    return {"nodes": len(nodes), "processed_scans": len(processed), "scans_per_s": len(processed) / best[0], "ms_per_scan": 1000 * best[0] / len(processed),
            "h2d_bytes_per_scan": int(np.mean([16 * len(v) for v in scans.values()])), "gpu_launches": int(best[1]), "final_map_points": int(best[2]),
            "cpu_oracle_scans_per_s": len(processed) / cpu_dt, "cpu_oracle_hot_path_share": hot / cpu_dt,
            "final_map_bit_identical_to_oracle": same,
            "quality_vs_initial_map": {"PR": round(pr["PR"], 3), "RR": round(pr["RR"], 3), "F1": round(pr["F1"], 4),
                                        "note": "erasor_b200/evaluate.py == reference scripts/analysis_runner.py metric; GT = labelled initial map (synthetic twin)"},
            "pass_ms": pass_ms, "cpu_oracle_pass_ms": round(1000 * cpu_dt, 1),
            "timing": "wall clock around the synchronous C-ABI calls, best of 5 passes (the first includes module load and buffer allocation); "
                      "every processed node's scan is handed to erasor_updater_prefetch_scan one node ahead (upload + voxelisation under the previous node's path)"}


def ncu_dram_traffic():
    """DRAM bytes per launch (read + write) of the node-mode step's kernels from the committed ncu capture of this workload."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02", "ncu_nodes_raw.csv")
    out = {}
    try:
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        ik, ir, iw = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        names = (("k1_rpod_bin", "k1_rpod_bin"), ("k2_srt_scatter", "k2_scatter"), ("k4_rgpf", "k4_rgpf_all_classes"))
        for r in rows[2:]:
            for pat, key in names:
                if pat in r[ik]:
                    out[key] = out.get(key, 0.0) + float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0)
    except Exception:
        return {}
    return {k: float(round(v)) for k, v in out.items()}


def clocks_sampler_start(gpu_index: int):
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        return subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(gpu_index)],
                                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return None


def clocks_sampler_stop(proc):
    if proc is None:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    proc.terminate()
    try:
        out, _ = proc.communicate(timeout=5)
    except Exception:
        proc.kill()
        out = ""
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in out.strip().splitlines():
        f = [x.strip() for x in line.split(",")]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0])); mx.append(float(f[1]))
        except ValueError:
            continue
        for nme, v in zip(names, f[3:7]):
            if v.lower().startswith("active"):
                reasons.add(nme)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
            "samples": len(sm), "reasons": sorted(reasons)}


def final_map_quality(map_world, keep):
    """NN-matched Preservation / Rejection rate (reference scripts/analysis.py:124-155 == erasor_b200/evaluate.py) of the
    static map this job produced: initial map minus every point some frame rejected."""
    from erasor_b200 import evaluate
    est = map_world[keep.astype(bool)]
    r = evaluate.evaluate(map_world, est)
    return {"PR": round(r["PR"], 3), "RR": round(r["RR"], 3), "F1": round(r["F1"], 4), "kept": int(keep.sum()), "of": int(len(keep))}


# ------------------------------------------------------------------------------------------------
# reference arm: the restated reference path (oracle port) on all host cores
# ------------------------------------------------------------------------------------------------
_W = {}


def _ref_init(pdict, map_world, poses, qs):
    from erasor_b200 import params
    from oracle import oracle_py
    _W["p"] = params.ErasorParams(**pdict)
    _W["o"] = oracle_py.Oracle(_W["p"])
    _W["fetch"] = oracle_py.fetch_voi
    _W["map"], _W["poses"], _W["qs"] = map_world, poses, qs


def _ref_node(i):
    voi, _ = _W["fetch"](_W["map"], _W["poses"][i], _W["p"].max_range)       # OfflineMapUpdater::fetch_VoI
    return _W["o"].run(voi, _W["qs"][i])                                       # set_inputs .. get_static_estimate


def usable_cores():
    """CPUs this process can actually use: the affinity mask capped by the cgroup CPU quota (a container that sees 128 CPUs
    with cpu.max = 16 CPUs is throttled to 16; more worker processes than that only add contention)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    note = f"{n} CPUs in the affinity mask"
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:   # cgroup v1
                q, per = float(f.read()), float(g.read())
                if q > 0:
                    quota = q / per
        except (OSError, ValueError):
            pass
    if quota is not None and quota < n:
        n = max(1, int(quota))
        note += f", cgroup quota {quota:g} CPUs"
    return n, note


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import dataclasses
    import multiprocessing as mp
    from oracle import oracle_py
    oracle_py.build()
    p, map_world, poses, qs = load_workload(args.config, 0, 1, args.frames)
    cores, cores_note = usable_cores()
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_ref_init, initargs=(dataclasses.asdict(p), map_world, poses, qs)) as pool:
        # a step = the 20-node pass repeated until every worker has ~4 nodes (balanced waves): the reference is
        # single-threaded, so "all the host threads it can use" means independent nodes in parallel processes
        reps = max(1, -(-4 * cores // len(qs)))
        idx = list(range(len(qs))) * reps
        for _ in range(args.warmup):
            pool.map(_ref_node, idx, chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_ref_node, idx, chunksize=1)
        dt = time.perf_counter() - t0
    sps = len(idx) * args.steps / dt
    nv = [len(oracle_py.fetch_voi(map_world, poses[i], p.max_range)[0]) for i in range(len(qs))]
    line = {
        "impl": "reference", "metric": "LiDAR scans/sec through R-POD+SRT+R-GPF on KITTI-05 (synthetic twin)",
        "value": sps, "unit": "scans/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 points, f64 index/SRT arithmetic", "data": "synthetic",
        "config": workload_config(args.config, p, len(map_world), nv, qs, 1),
        "cpu_baseline": {"value": sps, "unit": "scans/s", "cores": cores, "kind": "port",
                         "sample": f"{len(idx)} nodes per step x {args.steps} steps, one oracle process per usable core ({cores_note}); per node: "
                                   "fetch_VoI + set_inputs + compare + get_static_estimate, oracle -O2, v3 WITHOUT the in-bin voxelisation "
                                   "(skip_voxelize=1 on both arms: lighter than the shipped v3, erasor.cpp:526-528) "
                                   "(the reference itself is single-threaded and cannot be compiled here: needs ROS/PCL/Eigen)"},
        "e2e": {"value": sps, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(config, p, n_map, n_voi, qs, world):
    return {"workload": CONFIGS[config]["what"] + ", frame-independent pass against the resident map (erasor_process_nodes)",
            "frames_per_step_per_gpu": len(qs), "frames_per_step": len(qs) * world,
            "rings_x_sectors": f"{p.num_rings}x{p.num_sectors}", "max_range_m": p.max_range, "version": p.version,
            "map_points": int(n_map), "mean_map_voi_points": int(np.mean(n_voi)) if len(n_voi) else 0,
            "mean_query_points": int(np.mean([len(q) for q in qs])),
            "in_bin_voxelize": "skipped on both arms (skip_voxelize=1): v3's per-bin VoxelGrid only changes the cloud outputs, not the masks",
            "l2": f"resident arm: {N_QUERY_COPIES} rotating query copies (> 126 MB L2); the map is resident by design (uploaded once); "
                  "e2e arm: inputs come from host memory every step",
            "parallelism": f"frames sharded x{world} (strided: rank r takes nodes r, r + {world}, ...)"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from erasor_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: erasor_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")          # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)

    p, map_world, poses, qs = load_workload(args.config, rank, world, args.frames)
    F = len(qs)
    qo = np.cumsum([0] + [len(q) for q in qs]).astype(np.uint64)
    Q = np.ascontiguousarray(np.concatenate(qs), dtype=np.float32)
    NQ, NG = len(Q), len(map_world)

    t_up = time.perf_counter()
    gmap = capi.Map(map_world, device=local)                   # load_global_map: once per job, outside the timed steps
    map_upload_ms = 1000 * (time.perf_counter() - t_up)
    L = max(1, args.lanes)
    lanes = [capi.Handle(p, device=local) for _ in range(L)]
    for h in lanes:
        h.attach_map(gmap)
    h0 = lanes[0]
    xs = torch.cuda.ExternalStream(h0.stream, device=dev)

    n_copies = max(2, min(N_QUERY_COPIES, int(3e9 // max(1, 16 * NQ))))
    dQ = [torch.from_numpy(Q).to(dev) for _ in range(n_copies)]
    hQ = torch.from_numpy(Q).pin_memory()
    hQ3 = torch.from_numpy(np.ascontiguousarray(Q[:, :3])).pin_memory()      # packed x y z: the masks never read the query's intensity
    hK = [torch.empty(NG, dtype=torch.uint8).pin_memory() for _ in range(L)]
    torch.cuda.synchronize()

    # The path's one exchange (north_star): R-GPF's epilogue folds every frame's verdict onto the map's keep mask (a point
    # survives if no frame rejected it); the per-rank masks are bit-packed, all-gathered with ONE ncclAllGather over NVLink
    # and AND-ed by a library kernel (erasor_allgather_and_keep) -- all behind the C ABI, nothing of torch on the path.
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt = torch.frombuffer(bytearray(capi.comm_unique_id()), dtype=torch.uint8).to(dev)
        dist.broadcast(idt, 0)                                 # control plane: ships the 128-byte NCCL id
        h0.comm_init(bytes(idt.cpu().numpy().tobytes()), world, rank)

    def exchange():
        h0.allgather_and_keep(gmap.keep_ptr, NG)               # asynchronous on lane 0's stream; no-op at N=1

    def submit_resident(i, lane):
        lanes[lane].process_nodes_ptr(poses, dQ[i % n_copies].data_ptr(), qo, 0.0, 0, 0, capi.PTR_DEVICE, asynchronous=True)

    def submit_host(i, lane):
        lanes[lane].process_nodes_ptr(poses, hQ3.data_ptr(), qo, 0.0, 0, hK[lane].data_ptr(), capi.PTR_HOST | capi.PTR_QUERY_XYZ, asynchronous=True)

    def submit_host_xyzi(i, lane):
        lanes[lane].process_nodes_ptr(poses, hQ.data_ptr(), qo, 0.0, 0, hK[lane].data_ptr(), capi.PTR_HOST, asynchronous=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def wait_all():
        for h in lanes:
            h.wait()

    def timed(submit, steps, warmup, n_lanes):
        # every (lane, input copy) pair is seen once before the clock starts: the library captures one CUDA graph per distinct
        # set of buffer pointers, and a first use must not land inside the timed region
        warmup = max(warmup, n_copies * n_lanes if submit is submit_resident else n_lanes)
        for i in range(warmup):
            lanes[i % n_lanes].wait()
            submit(i, i % n_lanes)
        wait_all()
        exchange()                                 # the collective is warm before the timed region (NCCL connects lazily)
        h0.synchronize()
        gmap.reset_keep()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = sum(h.kernel_launch_count() for h in lanes)
        gc.disable()                               # a collection inside a 2 ms timed region would be most of it
        e0.record(xs)                              # every lane is idle here
        for i in range(steps):
            lane = i % n_lanes
            lanes[lane].wait()                     # a handle carries one submission at a time
            submit(warmup + i, lane)
        wait_all()
        gc.enable()
        e_steps = torch.cuda.Event(enable_timing=True)
        e_steps.record(xs)
        exchange()                                 # the job's one collective, inside the timed region
        e1.record(xs)
        barrier()
        ms, ms_steps = e0.elapsed_time(e1), e0.elapsed_time(e_steps)
        t = torch.tensor([ms, ms_steps], dtype=torch.float64, device=dev)
        per_rank = None
        if world > 1:
            allt = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            per_rank = [[round(float(x[0]), 4), round(float(x[1]), 4)] for x in allt]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0].item()), sum(h.kernel_launch_count() for h in lanes) - l0, per_rank

    sampler = clocks_sampler_start(local) if rank == 0 else None
    if sampler is not None:
        t_busy = time.perf_counter()
        i_busy = 0
        while time.perf_counter() - t_busy < 1.0:        # untimed: gives nvidia-smi (200 ms period, the recipe's; faster polling stalls the launches it shares the driver with) samples under this load
            lanes[i_busy % L].wait()
            submit_resident(i_busy, i_busy % L)
            i_busy += 1
        wait_all()
    W = max(args.warmup, 3)
    # --- per-kernel CUDA-event times: one lane, plain launches (events cannot be recorded inside a captured graph) ---
    h0.reset_kernel_times(True)
    ms_ev, _, _ = timed(submit_resident, args.steps, W, 1)
    kt = {name: h0.kernel_time_ms(i) for i, name in ((1, "k1_rpod_bin"), (2, "k2_scatter"), (3, "k3_srt"), (4, "k4_rgpf_all_classes"))}
    kernel_ms = {k: v[0] / max(1, v[1]) for k, v in kt.items()}
    h0.reset_kernel_times(False)
    # --- value: resident inputs, one lane (dependent steps) and `L` overlapped lanes ---
    # Every headline block of K steps is timed REPEATS times and the MEDIAN block is reported (all block times are in the line,
    # `blocks_ms`): a block lasts 2-4 ms, and a single host-side hiccup (an nvidia-smi poll holding the driver, a descheduled
    # launch thread) inside one would otherwise be the number.
    REPEATS = 3
    blocks = {}

    def timed_median(name, submit, n_lanes):
        runs = [timed(submit, args.steps, W, n_lanes) for _ in range(REPEATS)]
        blocks[name] = [round(r[0], 4) for r in runs]
        return sorted(runs, key=lambda r: r[0])[REPEATS // 2]

    ms_res_1, launches_1, _ = timed_median("resident_one_lane", submit_resident, 1)
    ms_res, launches, per_rank_res = timed_median("resident", submit_resident, L)
    # what the headline path handed its caller in its last timed step: the map's folded keep mask and that batch's per-node counters
    outputs = None
    if args.dump_outputs and rank == 0:
        n_voi_last, n_flag_last, n_rej_last = lanes[(args.steps - 1) % L].node_stats()
        outputs = {"map_keep": gmap.get_keep().astype(np.float32), "node_voi_points": n_voi_last.astype(np.float64),
                   "node_flagged_bins": n_flag_last.astype(np.float64), "node_rejected_points": n_rej_last.astype(np.float64)}
    # --- e2e: host buffers through the same call ---
    ms_e2e_1, _, _ = timed_median("e2e_one_lane", submit_host, 1)
    ms_e2e, _, per_rank_e2e = timed_median("e2e", submit_host, L)
    ms_e2e_xyzi, _, _ = timed(submit_host_xyzi, args.steps, W, L)
    clocks = clocks_sampler_stop(sampler) if rank == 0 else None

    # final static map of the job (untimed repeat of one step + exchange) and per-node counters
    gmap.reset_keep()
    dFK = torch.empty((F, NG), dtype=torch.uint8, device=dev)
    h0.process_nodes_ptr(poses, dQ[0].data_ptr(), qo, 0.0, dFK.data_ptr(), 0, capi.PTR_DEVICE)
    n_voi, n_flag, n_rej = h0.node_stats()
    npts_flagged, _ = h0.rgpf_profile()
    exchange()
    h0.synchronize()
    keep_final = gmap.get_keep()

    if rank == 0:
        from oracle import oracle_py
        oracle_py.build()
        # cpu_baseline: the oracle port on ONE core over a bounded sample of this workload
        o = oracle_py.Oracle(p)
        t0 = time.perf_counter()
        reps, nfr, t_voi = 0, 0, 0.0
        while True:
            for f in range(F):
                t1 = time.perf_counter()
                voi, idx = oracle_py.fetch_voi(map_world, poses[f], p.max_range)
                t_voi += time.perf_counter() - t1
                o.run(voi, qs[f])
                nfr += 1
            reps += 1
            if time.perf_counter() - t0 > 10.0 or reps >= 20:
                break
        cpu_dt = time.perf_counter() - t0
        # -O0 note (the reference's CMakeLists.txt:3-4 sets no optimisation level): one pass over the frames
        o0 = oracle_py.Oracle(p, opt="O0")
        t1 = time.perf_counter()
        n0 = 0
        for f in range(min(F, 6)):
            voi, _ = oracle_py.fetch_voi(map_world, poses[f], p.max_range)
            o0.run(voi, qs[f]); n0 += 1
        o0_sps = n0 / (time.perf_counter() - t1)
        # parity spot check of the benchmarked output (frame 0) against the oracle
        voi, idx = oracle_py.fetch_voi(map_world, poses[0], p.max_range)
        o.run(voi, qs[0])
        _, rej = o.cloud(o.MAP_REJECTED)
        ok0 = np.ones(NG, dtype=np.uint8)
        ok0[idx[rej]] = 0
        parity_ok = bool(np.array_equal(dFK[0].cpu().numpy(), ok0))

        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        NV, n_f = int(n_voi.sum()), int(npts_flagged.sum())
        scans = F * world
        value = scans * args.steps / (ms_res * 1e-3)
        # algorithmic bytes (SURVEY 8d): bytes_frame = 16 (N_m + N_q) + N_m + 16 N_F with N_m = the node's VoI; per kernel:
        # K1 in node mode is the FUSED fetch_VoI + binning kernel: SURVEY 8d's rule for it is 16 B per map point scanned (16 N_map_total
        # per frame) instead of 16 N_m; the unfused figure (VoI + query points only) is kept beside it as `frac_voi_bytes`
        kbytes = {"k1_rpod_bin": 16.0 * (F * NG + NQ),
                  "k2_scatter": 2.0 * 2 * F * NG + 36.0 * n_f,            # bin ids twice + 36 B per scattered point
                  "k3_srt": 36.0 * F * p.num_bins,
                  "k4_rgpf_all_classes": 16.0 * n_f + 4.0 * n_f + float(n_rej.sum())}
        by_kernel = {k: {"avg_launch_ms": round(kernel_ms[k], 5), "algorithmic_bytes_per_launch": kbytes[k],
                         "achieved_gbs": round(kbytes[k] / (kernel_ms[k] * 1e-3) / 1e9, 1) if kernel_ms[k] > 0 else 0.0,
                         "frac": round(kbytes[k] / (kernel_ms[k] * 1e-3) / 1e9 / peak, 4) if kernel_ms[k] > 0 else 0.0,
                         "share_of_event_timed_step": round(kernel_ms[k] / (ms_ev / args.steps), 3)} for k in kernel_ms}
        by_kernel["k1_rpod_bin"]["frac_voi_bytes"] = round(16.0 * (NV + NQ) / (kernel_ms["k1_rpod_bin"] * 1e-3) / 1e9 / peak, 4) if kernel_ms["k1_rpod_bin"] > 0 else 0.0
        by_kernel["k1_rpod_bin"]["note"] = ("fused fetch_VoI + R-POD: 16 B per map point scanned per frame (SURVEY 8d fused rule) + 16 B per query point; the resident map "
                                            "(16 N_map bytes) stays in the 126 MB L2 across the frames of a step, so DRAM traffic is far BELOW these bytes and the kernel is issue-bound")
        dom = max(kernel_ms, key=lambda k: kernel_ms[k])
        step_bytes = 16.0 * (NV + NQ) + NV + 16.0 * n_f
        step_ms = ms_res / args.steps
        step_gbs = step_bytes / (step_ms * 1e-3) / 1e9
        ncu_traffic = ncu_dram_traffic() if (args.config == "seq05" and F == FRAMES_PER_PASS) else {}
        line = {
            "metric": "LiDAR scans/sec through R-POD+SRT+R-GPF on KITTI-05 (synthetic twin)",
            "value": value, "unit": "scans/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 points, f64 index/SRT arithmetic", "data": "synthetic",
            "config": workload_config(args.config, p, NG, n_voi, qs, world),
            "blocks_ms": {"repeats": REPEATS, "reported": "median block", **blocks},
            "lanes": {"handles": L, "value_one_lane": scans * args.steps / (ms_res_1 * 1e-3), "ms_per_step_one_lane": ms_res_1 / args.steps,
                      "e2e_one_lane": scans * args.steps / (ms_e2e_1 * 1e-3),
                      "note": "asynchronous submissions round-robin over `handles` C-ABI handles sharing one resident map: a batch's "
                              "R-GPF (latency-bound) runs under the next batch's binning; one_lane = dependent steps"},
            "e2e": {"value": scans * args.steps / (ms_e2e * 1e-3), "unit": "scans/s",
                    "h2d_bytes_per_step": int(12 * NQ + 80 * F), "d2h_bytes_per_step": int(NG),
                    "value_xyzi_queries": scans * args.steps / (ms_e2e_xyzi * 1e-3), "h2d_bytes_per_step_xyzi_queries": int(16 * NQ + 80 * F),
                    "note": "pinned host poses + queries (packed x y z, ERASOR_PTR_QUERY_XYZ: the masks never read the query's intensity) -> "
                            "erasor_process_nodes_async(PTR_HOST) -> pinned host keep mask of the map, every step; value_xyzi_queries = the same "
                            "call with 16-byte x y z i queries; "
                            f"the map itself was uploaded once before the steps ({map_upload_ms:.1f} ms for {16 * NG} bytes, load_global_map)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": by_kernel[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                         "frac": by_kernel[dom]["frac"], "traffic": ncu_traffic.get(dom),
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": kbytes[dom], "avg_launch_ms": kernel_ms[dom],
                         "launches_timed": int(kt[dom][1]),
                         "why": "the dominant kernel by CUDA-event time (one lane, plain launches); by_kernel lists all of them: K1 moves the path's bytes "
                                "and is issue-bound, R-GPF is bound by a serial float dependency chain per bin (exact-order covariance sums + Jacobi SVD, "
                                "DESIGN.md section 5) and runs under the other kernels of overlapped submissions",
                         "hbm_kernel": "k1_rpod_bin", "by_kernel": by_kernel,
                         "traffic_by_kernel": ncu_traffic,
                         "traffic_source": "profiles/r02/ncu_nodes_raw.csv: dram__bytes_read.sum + dram__bytes_write.sum of one launch of each kernel on this "
                                           "workload (ncu --set full; the 5.4 MB map is L2-resident, so K1's DRAM traffic is far below the bytes it scans)",
                         "ms_per_step_with_event_timing": ms_ev / args.steps},
            "pipeline": {"bytes_per_step": step_bytes, "flagged_bin_points_per_step": n_f, "flagged_bins_per_step": int(len(npts_flagged)),
                         "achieved": step_gbs, "unit": "GB/s", "frac_of_hbm_peak": step_gbs / peak,
                         "frac_of_hbm_peak_one_lane": step_bytes / (ms_res_1 / args.steps * 1e-3) / 1e9 / peak},
            "cpu_baseline": {"value": nfr / cpu_dt, "unit": "scans/s", "cores": 1, "kind": "port",
                             "sample": f"{nfr} nodes ({reps} passes over this rank's {F}), oracle -O2, one core, per node fetch_VoI + ERASOR "
                                       f"(fetch_VoI share {t_voi / cpu_dt:.2f}); v3 without the in-bin voxelisation on both arms (skip_voxelize=1); "
                                       f"-O0 build (the reference's CMakeLists sets no -O level): {o0_sps:.1f} scans/s; "
                                       "reference cannot be compiled here (ROS/PCL/Eigen absent)"},
            "clocks": clocks,
            "parity_spot_check": parity_ok,
            "quality_final_map": dict(final_map_quality(map_world, keep_final),
                                      note="NN-matched PR/RR (scripts/analysis.py metric) of initial map minus every point some frame of the job rejected; "
                                           "GT = labelled initial map; compare offline_pass.quality_vs_initial_map (sequential reference mode)"),
            "exchange": {"comm_nranks": world, "collective": "one ncclAllGather of bit-packed masks + library AND kernel (erasor_allgather_and_keep), inside the timed region"
                         if world > 1 else "none (1 GPU)", "bytes_per_rank": int((NG + 31) // 32 * 4),
                         "per_rank_ms_total_and_steps_only": {"resident": per_rank_res, "e2e": per_rank_e2e}},
        }
        if world == 1 and args.config == "seq05" and not args.no_offline_pass:
            try:
                line["offline_pass"] = offline_pass_block(p, map_world, local)
            except Exception as e:      # the headline numbers must survive a failure of the informational block
                line["offline_pass"] = {"error": repr(e)}
        if world == 1 and args.config == "seq05" and not args.no_sweep:
            try:
                line["configs"] = {"3_seqs_00_01_02_07": sweep_presets(map_world, poses, qs, qo, dQ[0], gmap, local, args.steps),
                                   "4_large_scale_50M_voi": "profiles/r02/config4_largescale.json (scripts/config4_largescale.py)",
                                   "5_synthetic_40x360": "profiles/r02/config5_n*.json (bench.py --config synthetic40x360 --frames 32)"}
            except Exception as e:
                line["configs"] = {"error": repr(e)}
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
        print(json.dumps(line))
    for h in lanes:
        h.close()
    gmap.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def sweep_presets(map_world, poses, qs, qo, dQ, gmap, device, steps):
    """BASELINE config 3: the other KITTI yamls (seq 00 / 01 / 02 / 07 geometry and thresholds) back to back on the same twin:
    scans/s (resident, one lane, CUDA events) and the NN-matched PR/RR of the job's final map."""
    import torch
    from erasor_b200 import capi, params
    out = {}
    xs = None
    for name in ("seq_00", "seq_01", "seq_02", "seq_07"):
        p = params.preset(name).replace(skip_voxelize=1)
        h = capi.Handle(p, device=device)
        h.attach_map(gmap)
        xs = torch.cuda.ExternalStream(h.stream)
        for _ in range(3):
            h.process_nodes_ptr(poses, dQ.data_ptr(), qo, 0.0, 0, 0, capi.PTR_DEVICE)
        gmap.reset_keep()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(xs)
        for _ in range(steps):
            h.process_nodes_ptr(poses, dQ.data_ptr(), qo, 0.0, 0, 0, capi.PTR_DEVICE, asynchronous=True)
        h.wait()
        e1.record(xs)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        nv, nf, nr = h.node_stats()
        q = final_map_quality(map_world, gmap.get_keep())
        out[name] = {"rings_x_sectors": f"{p.num_rings}x{p.num_sectors}", "max_range_m": p.max_range, "scans_per_s": len(qs) / (ms * 1e-3),
                     "ms_per_step": ms, "mean_voi_points": int(nv.mean()), "flagged_bins_per_step": int(nf.sum()), "PR": q["PR"], "RR": q["RR"], "F1": q["F1"]}
        h.close()
    gmap.reset_keep()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_PASS, help="frames per step per GPU")
    ap.add_argument("--lanes", type=int, default=4, help="C-ABI handles fed round-robin (overlapped batches)")
    ap.add_argument("--config", default="seq05", choices=sorted(CONFIGS))
    ap.add_argument("--no-offline-pass", action="store_true", help="skip the informational sequential-pass block")
    ap.add_argument("--no-sweep", action="store_true", help="skip the config-3 preset sweep block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (map keep mask, per-node counters) "
                    "as DIR/<name>.npy, to compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
