"""GPU parity of node mode on raw scans (erasor_process_scans) and of save_static_map on the attached map, against the
oracle's reference-faithful query preparation: transform(voxelize_preserving_labels(scan, leaf), lidar2body) -> fetch_VoI ->
ERASOR, per node, on the same initial map.  Masks, node counters, the voxelised queries themselves (bit for bit, in voxel-key
order), batch edge cases in one submission, packed x y z, pinned host vs device pointers, the internal sub-batch split,
asynchronous lanes sharing one map, and pipeline.run_frame_independent end to end."""
import numpy as np
import pytest

from erasor_b200 import params as P
from test_frame_independent import OracleNodeMode, oracle_query

pytestmark = pytest.mark.gpu

L2B = [0.0, 0.0, 1.73, 0.0, 0.0, 0.0, 1.0]
# a lidar2body with a rotation: yaw 30 deg, pitch 2 deg, and an offset
_q = np.array([np.sin(np.deg2rad(1.0)) * np.cos(np.deg2rad(15.0)), np.sin(np.deg2rad(1.0)), np.sin(np.deg2rad(15.0)), np.cos(np.deg2rad(15.0))])
_q /= np.linalg.norm(_q)
L2B_ROT = [0.31, -0.12, 1.73] + list(_q)


@pytest.fixture(scope="module")
def capi():
    from erasor_b200 import capi as C
    return C


def _raw(small_workload, picks):
    scene = small_workload["scene"]
    ks = [small_workload["frames"][i][2] for i in picks]
    poses = np.stack([scene.pose7(k) for k in ks]).astype(np.float64)
    scans = [scene.scan(k, n_beams=32, n_az=900, seed_offset=17) for k in ks]
    return poses, scans


def _cat(scans):
    off = np.cumsum([0] + [len(s) for s in scans]).astype(np.uint64)
    return (np.concatenate(scans) if off[-1] else np.zeros((0, 4), np.float32)), off


def _xyz_bits(a):
    return np.ascontiguousarray(a[:, :3], dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("name,version", [("seq_05", 3), ("seq_05", 2), ("seq_00", 3), ("synthetic_40x360", 3)])
def test_process_scans_parity(capi, oracle_mod, small_workload, name, version):
    p = P.preset(name).replace(skip_voxelize=1, version=version)
    map_world = small_workload["map_world"]
    poses, scans = _raw(small_workload, range(6))
    S, so = _cat(scans)
    o = OracleNodeMode(oracle_mod, None, p, map_world)
    o.process_scans(poses, S, so, 0.2, L2B, p.max_range)
    ofk, ost = np.stack(o.frame_keep), np.array(o.stats, dtype=np.int64)
    assert (ofk == 0).any(), "the workload must reject something"
    m = capi.Map(map_world)
    h = capi.Handle(p)
    h.attach_map(m)
    for rep in range(2):                       # second call: descriptors and graph reused
        m.reset_keep()
        keep, fk = h.process_scans(poses, S, so, 0.2, L2B, want_frame_keep=True)
        assert np.array_equal(fk, ofk), f"{name} v{version}: per-frame masks differ in {np.count_nonzero(fk != ofk)} points"
        assert np.array_equal(keep, ofk.min(axis=0)) and np.array_equal(m.get_keep(), keep)
    nv, nf, nr = h.node_stats()
    assert np.array_equal(nv, ost[:, 0]) and np.array_equal(nf, ost[:, 1]) and np.array_equal(nr, ost[:, 2])
    # the queries themselves: bit-identical to the reference's voxelised, transformed scans, in voxel-key order
    xyz, qoff = h.scan_queries()
    for f, q in enumerate(o.queries):
        assert np.array_equal(xyz[int(qoff[f]):int(qoff[f + 1])].view(np.uint32), _xyz_bits(q)), f"frame {f} query"
    # process_nodes fed those queries gives the same masks
    m.reset_keep()
    Q = np.concatenate(o.queries)
    keep2, fk2 = h.process_nodes(poses, Q, np.cumsum([0] + [len(q) for q in o.queries]).astype(np.uint64), want_frame_keep=True)
    assert np.array_equal(fk2, ofk) and np.array_equal(keep2, keep)
    h.close(); m.close()


def test_scan_queries_equal_the_updaters_query(capi, oracle_mod, small_workload):
    """The batched voxeliser and the sequential updater's (one scan per launch) produce the same QUERY_VOI."""
    p = P.preset("seq_05")
    up = P.updater_preset("seq_05")
    up.removal_interval = 1
    up.lidar2body = list(L2B_ROT)
    map_world = small_workload["map_world"]
    poses, scans = _raw(small_workload, range(3))
    u = capi.Updater(up, p, map_world)
    m = capi.Map(map_world)
    h = capi.Handle(p)
    h.attach_map(m)
    S, so = _cat(scans)
    h.process_scans(poses, S, so, up.query_voxel_size, up.lidar2body)
    xyz, qoff = h.scan_queries()
    for f in range(3):
        assert u.process_node(f + 1, poses[f], scans[f])
        uq = u.cloud(u.QUERY_VOI)
        assert np.array_equal(xyz[int(qoff[f]):int(qoff[f + 1])].view(np.uint32), _xyz_bits(uq)), f
        assert np.array_equal(_xyz_bits(uq), _xyz_bits(oracle_query(oracle_mod, scans[f], up.query_voxel_size, up.lidar2body)))
    u.close(); h.close(); m.close()


def _edge_scans(small_workload):
    scene = small_workload["scene"]
    rng = np.random.default_rng(11)
    big = scene.scan(small_workload["frames"][2][2], n_beams=128, n_az=2200, seed_offset=3)            # ~250 k points
    small = scene.scan(small_workload["frames"][1][2], n_beams=32, n_az=900)[:100]
    far = np.concatenate([rng.uniform(-4.0e4, 4.0e4, (3000, 3)), rng.integers(0, 300, (3000, 1))], axis=1).astype(np.float32)   # grid overflows int32
    mid = scene.scan(small_workload["frames"][4][2], n_beams=32, n_az=900, seed_offset=5)
    empty = np.zeros((0, 4), np.float32)
    return [mid, empty, far, small, big, empty, mid[::3].copy()]


@pytest.mark.parametrize("leaf", [0.05, 0.2, 0.5])
def test_batch_edges_in_one_submission(capi, oracle_mod, small_workload, leaf):
    import torch
    p = P.preset("seq_05").replace(skip_voxelize=1)
    map_world = small_workload["map_world"]
    scans = _edge_scans(small_workload)
    assert len(scans[4]) > 200000
    poses = np.stack([small_workload["scene"].pose7(small_workload["frames"][i % 6][2]) for i in range(len(scans))]).astype(np.float64)
    S, so = _cat(scans)
    m = capi.Map(map_world)
    h = capi.Handle(p)
    h.attach_map(m)
    keep, fk = h.process_scans(poses, S, so, leaf, L2B_ROT, want_frame_keep=True)
    xyz, qoff = h.scan_queries()
    for f, s in enumerate(scans):
        q = oracle_query(oracle_mod, s, leaf, L2B_ROT)
        assert np.array_equal(xyz[int(qoff[f]):int(qoff[f + 1])].view(np.uint32), _xyz_bits(q)), f"leaf {leaf} frame {f}"
    assert qoff[2] - qoff[1] == 0 and qoff[3] - qoff[2] == len(scans[2])            # empty; overflow returned unfiltered
    # the masks equal process_nodes on those queries (itself checked against the oracle in test_gpu_nodes.py)
    m.reset_keep()
    Q = np.concatenate([oracle_query(oracle_mod, s, leaf, L2B_ROT) for s in scans])
    keep_n, fk_n = h.process_nodes(poses, Q, qoff, want_frame_keep=True)
    assert np.array_equal(fk, fk_n) and np.array_equal(keep, keep_n)
    # packed x y z == x y z i
    m.reset_keep()
    keep_x, fk_x = h.process_scans(poses, S, so, leaf, L2B_ROT, want_frame_keep=True, packed_xyz=True)
    assert np.array_equal(fk_x, fk) and np.array_equal(keep_x, keep)
    xyz_x, qoff_x = h.scan_queries()
    assert np.array_equal(qoff_x, qoff) and np.array_equal(xyz_x.view(np.uint32), xyz.view(np.uint32))
    # pinned host pointers == device pointers (packed, at a 4-byte-aligned address), asynchronous
    sp = capi.scan_params(leaf, L2B_ROT)
    hS = torch.from_numpy(S).pin_memory()
    hK = torch.empty(len(map_world), dtype=torch.uint8).pin_memory()
    dS3 = torch.zeros(3 * len(S) + 1, dtype=torch.float32, device="cuda")
    dS3[1:] = torch.from_numpy(np.ascontiguousarray(S[:, :3])).cuda().reshape(-1)
    dK = torch.empty(len(map_world), dtype=torch.uint8, device="cuda")
    dFK = torch.empty((len(scans), len(map_world)), dtype=torch.uint8, device="cuda")
    for rep in range(2):
        m.reset_keep()
        h.process_scans_ptr(sp, poses, hS.data_ptr(), so, 0.0, 0, hK.data_ptr(), capi.PTR_HOST, asynchronous=True)
        h.wait()
        assert np.array_equal(hK.numpy(), keep), rep
        m.reset_keep()
        h.process_scans_ptr(sp, poses, dS3.data_ptr() + 4, so, 0.0, dFK.data_ptr(), dK.data_ptr(), capi.PTR_DEVICE | capi.PTR_QUERY_XYZ, asynchronous=True)
        h.wait()
        assert np.array_equal(dK.cpu().numpy(), keep) and np.array_equal(dFK.cpu().numpy(), fk), rep
    h.close(); m.close()


def test_invalid_arguments(capi, small_workload):
    p = P.preset("seq_05")
    m = capi.Map(small_workload["map_world"])
    h = capi.Handle(p)
    h.attach_map(m)
    poses, scans = _raw(small_workload, [0])
    S, so = _cat(scans)
    for leaf, l2b in ((0.0, L2B), (-0.2, L2B), (float("nan"), L2B), (0.2, [0, 0, 0, 0, 0, 0, 0]), (0.2, [float("inf")] + L2B[1:])):
        with pytest.raises(capi.ErasorError) as e:
            h.process_scans(poses, S, so, leaf, l2b)
        assert e.value.code == capi.E_INVALID
    with pytest.raises(capi.ErasorError) as e:
        h.process_scans(poses, S, np.array([5, 0], dtype=np.uint64), 0.2, L2B)
    assert e.value.code == capi.E_INVALID
    bad = poses.copy(); bad[0, 0] = np.nan
    with pytest.raises(capi.ErasorError) as e:
        h.process_scans(bad, S, so, 0.2, L2B)
    assert e.value.code == capi.E_INVALID
    with pytest.raises(capi.ErasorError):
        h.save_static_map(0.0)
    h.close(); m.close()


def test_sub_batch_split_and_lanes(capi, oracle_mod, small_workload):
    """150 scans with 40 x 360 bins is more than one submission's work queue (145 frames): split internally; and three
    asynchronous lanes sharing one map give the AND of their verdicts."""
    p = P.preset("synthetic_40x360").replace(skip_voxelize=1)
    map_world = small_workload["map_world"]
    scene = small_workload["scene"]
    base = [scene.scan(small_workload["frames"][i][2], n_beams=32, n_az=900, seed_offset=17) for i in range(6)]
    poses = np.stack([scene.pose7(small_workload["frames"][i % 6][2]) for i in range(150)]).astype(np.float64)
    scans = [base[i % 6] for i in range(150)]
    S, so = _cat(scans)
    m = capi.Map(map_world)
    h = capi.Handle(p)
    h.attach_map(m)
    keep, fk = h.process_scans(poses, S, so, 0.2, L2B, want_frame_keep=True)
    Q = [oracle_query(oracle_mod, s, 0.2, L2B) for s in base]
    m.reset_keep()
    keep_n, fk_n = h.process_nodes(poses, np.concatenate([Q[i % 6] for i in range(150)]),
                                   np.cumsum([0] + [len(Q[i % 6]) for i in range(150)]).astype(np.uint64), want_frame_keep=True)
    assert np.array_equal(fk, fk_n) and np.array_equal(keep, keep_n) and (keep == 0).any()
    h.close()
    # lanes
    import torch
    p5 = P.preset("seq_05").replace(skip_voxelize=1)
    poses6, scans6 = _raw(small_workload, range(6))
    o = OracleNodeMode(oracle_mod, None, p5, map_world)
    o.process_scans(poses6, *_cat(scans6), 0.2, L2B, p5.max_range)
    sp = capi.scan_params(0.2, L2B)
    lanes = []
    for g in ([0, 1], [2, 3], [4, 5]):
        Sg, sog = _cat([scans6[i] for i in g])
        hh = capi.Handle(p5)
        hh.attach_map(m)
        lanes.append(dict(h=hh, poses=np.ascontiguousarray(poses6[g]), so=sog, dS=torch.from_numpy(Sg).cuda(), hS=torch.from_numpy(Sg).pin_memory()))
    torch.cuda.synchronize()
    for kind in ("device", "host"):
        for rep in range(3):
            m.reset_keep()
            for L in lanes:
                ptr, pk = (L["dS"].data_ptr(), capi.PTR_DEVICE) if kind == "device" else (L["hS"].data_ptr(), capi.PTR_HOST)
                L["h"].process_scans_ptr(sp, L["poses"], ptr, L["so"], 0.0, 0, 0, pk, asynchronous=True)
            for L in lanes:
                L["h"].wait()
            assert np.array_equal(m.get_keep(), o.keep), (kind, rep)
    for L in lanes:
        L["h"].close()
    m.close()


@pytest.mark.parametrize("leaf", [0.05, 0.2])
def test_save_static_map(capi, oracle_mod, small_workload, leaf):
    p = P.preset("seq_05").replace(skip_voxelize=1)
    map_world = small_workload["map_world"]
    poses, scans = _raw(small_workload, range(6))
    m = capi.Map(map_world)
    h = capi.Handle(p)
    h.attach_map(m)
    S, so = _cat(scans)
    keep, _ = h.process_scans(poses, S, so, 0.2, L2B)
    assert (keep == 0).any()
    got = h.save_static_map(leaf)
    expect = oracle_mod.voxelize(map_world[keep == 1], leaf)
    assert got.shape == expect.shape and np.array_equal(got.view(np.uint32), expect.view(np.uint32))
    m.reset_keep()
    full = h.save_static_map(leaf)
    assert np.array_equal(full.view(np.uint32), oracle_mod.voxelize(map_world, leaf).view(np.uint32))
    h.close(); m.close()


def test_run_frame_independent_device_equals_stand_in(oracle_mod, small_workload):
    from erasor_b200 import pipeline
    ep = P.preset("seq_05")
    up = P.updater_preset("seq_05")
    up.removal_interval = 2
    scene = small_workload["scene"]
    nodes = [(k, scene.pose7(k), scene.scan(k, n_beams=32, n_az=900)) for k in range(0, 40, 2)]
    map_world = small_workload["map_world"]
    dev = pipeline.run_frame_independent(nodes, map_world, up, ep, nodes_per_step=4)
    ref = pipeline.run_frame_independent(nodes, map_world, up, ep, nodes_per_step=4, make_handle=lambda u, e, m: OracleNodeMode(oracle_mod, u, e, m))
    assert dev["processed_scans"] == ref["processed_scans"] == 10
    assert np.array_equal(dev["static_map"].view(np.uint32), ref["static_map"].view(np.uint32))
    assert dev["quality"] == ref["quality"]
