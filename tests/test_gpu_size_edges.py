"""GPU parity at every size where a kernel switches code path, against the CPU oracle, bit for bit.

- R-GPF (K4) size classes and sort networks: 128 / 256 / 384 / 512 (class A), 1024 / 1536 / 2048 / 2560 (class B, radix above
  2048), 2561 (class C), and class C's switch from shared memory to its slice of the global scratch above 8775 points.
- Several class-C global-scratch bins next to each other in source order, running with class A and B bins.
- K4b in-bin voxelisation (version 3): shared memory up to qc + ng = 4549 points, global scratch above; an int32-overflowing
  VoxelGrid; keys that need four 8-bit passes.
- K2's slot windows (40 x 360 bins): frames with one window less one slot, exactly one window, one slot more, two windows and
  one slot, and nearly all bins flagged, in mask mode and node mode.
- The batched voxeliser's cloud digits: more than 512 clouds in one submission take a second cloud digit, and the total crosses
  the radix-sort segment-length switch at 2 097 152 points.

Each test asserts that it hit its edge (bin sizes from the oracle's binning, qc + ng, flagged-bin counts, the number of scans in
one submission)."""
import numpy as np
import pytest

from crafted_bins import BinSpec, Z_KINDS, bin_id, crafted_frame, single_bin_frame
from erasor_b200 import params as P

pytestmark = pytest.mark.gpu

RGPF_SIZES = [128, 129, 256, 257, 384, 385, 512, 513, 1024, 1025, 1536, 1537, 2048, 2049, 2560, 2561, 8775, 8776, 30000, 120000]
K4C_SMEM_CAP = ((180 * 1024) - 32) // 21         # launch_k4_class<1024, 1024>: class-C bins above this use the global scratch
K4B_SMEM_CAP = (160 * 1024 - 64) // 36            # launch_k4b: in-bin voxelisation above this uses the global scratch
NODE_SPACING = 256.0                              # node mode: frame f is placed at x + 256 f (more than two VoI radii apart)
L2B = [0.0, 0.0, 1.73, 0.0, 0.0, 0.0, 1.0]


def k2_window(B, W=8):
    """k2_smem_plan: slot window of the flagged-bin scatter (mask and node mode)"""
    fixed = (2 * (B + 2) + 15) & ~15
    full = 4 * (W + 1) * B + fixed
    budget = full if full <= 111 * 1024 else 111 * 1024
    return min(max(B, 1), max(1, (budget - fixed) // (4 * (W + 1))))


@pytest.fixture(scope="module")
def capi():
    from erasor_b200 import capi as C
    return C


def _rejected_mask(o, n):
    _, rej = o.cloud(o.MAP_REJECTED)
    k = np.ones(n, dtype=np.uint8)
    k[rej] = 0
    return k


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _cloud_parity(capi, oracle_mod, p, m, q):
    """cloud mode, one frame: planes, static estimate and outliers against the oracle; returns the oracle"""
    o = oracle_mod.Oracle(p)
    o.run(m, q)
    h = capi.Handle(p)
    h.set_inputs(m, q)
    h.compare(p.version)
    gp, op = h.get_planes(), o.planes()
    assert [g["bin"] for g in gp] == [x["bin"] for x in op]
    for g, x in zip(gp, op):
        assert (g["n_points"], g["n_seeds"], g["lpr"]) == (x["n_points"], x["n_seeds"], x["lpr"]), x["bin"]
        assert np.array_equal(g["normal_d"], x["normal_d"]) and np.array_equal(g["n_ground"], x["n_ground"]), x["bin"]
    arr, cmp_ = h.get_static_estimate()
    oarr, _ = o.cloud(o.ARRANGED)
    ocmp, _ = o.cloud(o.COMPLEMENT)
    assert arr.shape == oarr.shape and np.array_equal(_bits(arr), _bits(oarr)), "arranged"
    assert cmp_.shape == ocmp.shape and np.array_equal(_bits(cmp_), _bits(ocmp)), "complement"
    mr, cr = h.get_outliers()
    omr, _ = o.cloud(o.MAP_REJECTED)
    ocr, _ = o.cloud(o.CURR_REJECTED)
    assert mr.shape == omr.shape and np.array_equal(_bits(mr), _bits(omr)), "map rejected"
    assert cr.shape == ocr.shape and np.array_equal(_bits(cr), _bits(ocr)), "curr rejected"
    keep, _ = h.get_static_mask()
    assert np.array_equal(keep, _rejected_mask(o, len(m)))
    h.close()
    return o


def _mask_mode(capi, oracle_mod, p, frames):
    """process_frames over all frames in one batch: keep masks and frame_stats against the oracle; returns nf"""
    mo = np.cumsum([0] + [len(m) for m, _ in frames]).astype(np.uint64)
    qo = np.cumsum([0] + [len(q) for _, q in frames]).astype(np.uint64)
    h = capi.Handle(p)
    keep = h.process_frames(np.concatenate([m for m, _ in frames]), mo, np.concatenate([q for _, q in frames]), qo)
    nf, nr = h.frame_stats()
    h.close()
    o = oracle_mod.Oracle(p)
    for f, (m, q) in enumerate(frames):
        o.run(m, q)
        ok = _rejected_mask(o, len(m))
        assert np.array_equal(keep[int(mo[f]):int(mo[f + 1])], ok), f"mask mode, frame {f}: {np.count_nonzero(keep[int(mo[f]):int(mo[f + 1])] != ok)} points differ"
        assert (nf[f], nr[f]) == (len(o.planes()), int(np.count_nonzero(ok == 0))), f"mask mode, frame {f}"
    o.close()
    return nf


def _node_mode(capi, oracle_mod, p, frames):
    """process_nodes on one resident map that holds every frame (frame f moved to x + 256 f, its pose there): per-frame masks and
    node_stats against the oracle's fetch_VoI + ERASOR; returns nf"""
    shift = [np.array([NODE_SPACING * f, 0.0, 0.0, 0.0], dtype=np.float32) for f in range(len(frames))]
    mw = np.concatenate([m + shift[f] for f, (m, _) in enumerate(frames)]).astype(np.float32)
    poses = np.array([[NODE_SPACING * f, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0] for f in range(len(frames))], dtype=np.float64)
    qs = [q for _, q in frames]
    gm = capi.Map(mw)
    h = capi.Handle(p)
    h.attach_map(gm)
    keep, fk = h.process_nodes(poses, np.concatenate(qs), np.cumsum([0] + [len(q) for q in qs]).astype(np.uint64), want_frame_keep=True)
    nv, nf, nr = h.node_stats()
    h.close(); gm.close()
    o = oracle_mod.Oracle(p)
    for f in range(len(frames)):
        voi, idx = oracle_mod.fetch_voi(mw, poses[f], p.max_range)
        assert len(voi) == len(frames[f][0])
        o.run(voi, qs[f])
        _, rej = o.cloud(o.MAP_REJECTED)
        ok = np.ones(len(mw), dtype=np.uint8)
        ok[idx[rej]] = 0
        assert np.array_equal(fk[f], ok), f"node mode, frame {f}: {np.count_nonzero(fk[f] != ok)} points differ"
        assert (nv[f], nf[f], nr[f]) == (len(voi), len(o.planes()), len(rej)), f"node mode, frame {f}"
    assert np.array_equal(keep, fk.min(axis=0))
    o.close()
    return nf


def _bin_size(o, which, b):
    return int(np.count_nonzero(o.bin_of_point(which) == b))


# ---------------------------------------------------------------------------------------------------------------------------
# 1a. R-GPF size classes, sort networks and the class-C global scratch
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("z_kind", Z_KINDS)
def test_rgpf_size_edges(capi, oracle_mod, z_kind):
    assert K4C_SMEM_CAP == 8775
    p = P.preset("seq_05").replace(skip_voxelize=1, version=3)
    sizes = [n for n in RGPF_SIZES if n <= K4C_SMEM_CAP + 1 or z_kind in ("rough", "dup")]
    b = bin_id(p, 5, 2)
    frames = []
    for n in sizes:
        m, q = single_bin_frame(n, z_kind, 1000 + n, p)
        o = _cloud_parity(capi, oracle_mod, p, m, q)
        assert _bin_size(o, 0, b) == n, "the bin must hold exactly n map points"
        assert [x["n_points"] for x in o.planes()] == [n], "the crafted bin must be the one flagged bin"
        o.close()
        frames.append((m, q))
    assert np.array_equal(_mask_mode(capi, oracle_mod, p, frames), np.ones(len(frames)))
    assert np.array_equal(_node_mode(capi, oracle_mod, p, frames), np.ones(len(frames)))


# ---------------------------------------------------------------------------------------------------------------------------
# 1b. several class-C global-scratch bins next to each other, with class A and B bins running at the same time
# ---------------------------------------------------------------------------------------------------------------------------
def test_rgpf_adjacent_global_scratch_bins(capi, oracle_mod):
    p = P.preset("seq_05").replace(skip_voxelize=1, version=3)
    layouts = [
        [BinSpec(5, 2, 30000), BinSpec(6, 2, 12000), BinSpec(7, 2, 9000), BinSpec(5, 4, 300), BinSpec(5, 6, 2000)],
        [BinSpec(3, 10, 300, "dup"), BinSpec(4, 10, 20000, "dup"), BinSpec(5, 10, 8776, "dup"), BinSpec(6, 10, 1500, "dup"),
         BinSpec(8, 10, 9500, "dup"), BinSpec(9, 10, 2561)],
    ]
    frames = []
    for i, specs in enumerate(layouts):
        m, q = crafted_frame(np.random.default_rng(50 + i), p, specs)
        o = _cloud_parity(capi, oracle_mod, p, m, q)
        for s in specs:
            assert _bin_size(o, 0, bin_id(p, s.ring, s.sector)) == s.n
        assert sorted(x["n_points"] for x in o.planes()) == sorted(s.n for s in specs)
        assert sum(x["n_points"] > K4C_SMEM_CAP for x in o.planes()) >= 2
        o.close()
        frames.append((m, q))
    assert np.array_equal(_mask_mode(capi, oracle_mod, p, frames), [len(s) for s in layouts])
    assert np.array_equal(_node_mode(capi, oracle_mod, p, frames), [len(s) for s in layouts])


# ---------------------------------------------------------------------------------------------------------------------------
# 1c. K4b in-bin voxelisation: shared memory / global scratch, int32 overflow, four key passes
# ---------------------------------------------------------------------------------------------------------------------------
def _k4b_frame(oracle_mod, p, specs, targets, seed):
    """a frame whose flagged bins have qc + ng == target: R-GPF's ground count does not depend on the query, so one oracle run
    with a few query points gives ng, and the query counts follow"""
    o = oracle_mod.Oracle(p)
    o.run(*crafted_frame(np.random.default_rng(seed), p, specs))
    ng = {x["bin"]: int(x["n_ground"][-1]) for x in o.planes()}
    qc = [t - ng[bin_id(p, s.ring, s.sector)] for s, t in zip(specs, targets)]
    assert min(qc) >= 40
    m, q = crafted_frame(np.random.default_rng(seed), p, specs, query_counts=qc)
    o.run(m, q)
    for s, t in zip(specs, targets):
        b = bin_id(p, s.ring, s.sector)
        ngb = [int(x["n_ground"][-1]) for x in o.planes() if x["bin"] == b]
        assert len(ngb) == 1 and int(o.bins(1)[2][b]) + ngb[0] == t, f"bin {b}: qc + ng must be {t}"
    o.close()
    return m, q


def _cells(pts, leaf):
    """pcl::VoxelGrid's grid of a bin's K4b input, in float as the kernel computes it: (overflow, cell count)"""
    mn, mx = pts[:, :3].min(axis=0), pts[:, :3].max(axis=0)
    inv = np.float32(1.0) / np.float32(leaf)
    d = [int(np.float32(np.float32(mx[k] - mn[k]) * inv)) + 1 for k in range(3)]
    div = [int(np.floor(np.float32(mx[k] * inv))) - int(np.floor(np.float32(mn[k] * inv))) + 1 for k in range(3)]
    return d[0] * d[1] * d[2] > 2147483647, div[0] * div[1] * div[2]


def test_k4b_size_edges(capi, oracle_mod):
    assert K4B_SMEM_CAP == 4549
    p = P.preset("seq_05").replace(skip_voxelize=0, version=3)
    # 4549 stays in shared memory; 4550 and ~20 000 are two global-scratch bins next to each other in bin order
    specs = [BinSpec(5, 2, 3000), BinSpec(6, 2, 3000), BinSpec(7, 2, 12000)]
    m, q = _k4b_frame(oracle_mod, p, specs, [4549, 4550, 20000], seed=71)
    _cloud_parity(capi, oracle_mod, p, m, q).close()
    assert np.array_equal(_mask_mode(capi, oracle_mod, p, [(m, q)]), [3])
    assert np.array_equal(_node_mode(capi, oracle_mod, p, [(m, q)]), [3])


@pytest.mark.parametrize("leaf,edge", [(1e-4, "overflow"), (0.004, "four passes")])
def test_k4b_voxel_grid_edges(capi, oracle_mod, leaf, edge):
    p = P.preset("seq_05").replace(skip_voxelize=0, version=3, map_voxel_size=leaf)
    specs = [BinSpec(5, 2, 3000), BinSpec(6, 2, 3000)]
    m, q = _k4b_frame(oracle_mod, p, specs, [3000, 4600], seed=72)
    o = _cloud_parity(capi, oracle_mod, p, m, q)
    gv, _ = o.cloud(o.GROUND_VIZ)
    for s in specs:
        b = bin_id(p, s.ring, s.sector)
        inp = np.concatenate([q[o.bin_of_point(1) == b], gv[_bins_of(p, gv) == b]])      # K4b's input: bin_curr + ground
        ovf, cells = _cells(inp, leaf)
        if edge == "overflow":
            assert ovf, f"bin {b}: the VoxelGrid must overflow int32"
        else:
            assert not ovf and (1 << 24) < cells < (1 << 31), f"bin {b}: {cells} cells, the key must need four 8-bit passes"
    o.close()


def _bins_of(p, pts):
    from np_restatement import bin_of_points
    return bin_of_points(p, pts)[0]


# ---------------------------------------------------------------------------------------------------------------------------
# 1d. K2 slot windows
# ---------------------------------------------------------------------------------------------------------------------------
def _many_bins_frame(p, bins, seed):
    """every bin of `bins`: 8 ground + 4 object map points (map height span > 0.5) and 7 flat query points, well inside it"""
    rng = np.random.default_rng(seed)
    R = p.num_rings
    ring, sector = bins % R, bins // R

    def pts(k, lo, hi):
        rr, ss = np.repeat(ring, k), np.repeat(sector, k)
        r = (rr + rng.uniform(lo, hi, len(rr))) * (p.max_range / R)
        th = (ss + rng.uniform(lo, hi, len(ss))) * (2.0 * np.pi / p.num_sectors)
        return r * np.cos(th), r * np.sin(th)

    gx, gy = pts(8, 0.3, 0.7)
    g = np.stack([gx, gy, rng.normal(-0.9, 0.02, len(gx)), np.full(len(gx), 40.0)], axis=1)
    ox, oy = pts(4, 0.35, 0.65)
    oz = rng.uniform(-0.5, 1.0, (len(bins), 4))
    oz[:, 0] = 1.0
    ob = np.stack([ox, oy, oz.reshape(-1), np.full(len(ox), 252.0)], axis=1)
    qx, qy = pts(7, 0.3, 0.7)
    qq = np.stack([qx, qy, rng.uniform(-0.95, -0.85, len(qx)), np.full(len(qx), 40.0)], axis=1)
    m = rng.permutation(np.concatenate([g, ob])).astype(np.float32)
    return np.ascontiguousarray(m), np.ascontiguousarray(rng.permutation(qq).astype(np.float32))


def test_k2_slot_windows(capi, oracle_mod):
    p = P.preset("synthetic_40x360").replace(skip_voxelize=1, version=3)
    B = p.num_bins
    SW = k2_window(B)
    assert SW == 2356
    targets = [SW - 1, SW, SW + 1, 2 * SW + 1, B - 400]
    order = np.random.default_rng(3).permutation(B)
    frames = []
    for i, t in enumerate(targets):
        m, q = _many_bins_frame(p, np.sort(order[:t]), seed=300 + i)
        o = oracle_mod.Oracle(p)
        o.run(m, q)
        assert len(o.planes()) == t, f"frame {i}: {len(o.planes())} flagged bins, want {t}"
        o.close()
        frames.append((m, q))
    for nf in (_mask_mode(capi, oracle_mod, p, frames), _node_mode(capi, oracle_mod, p, frames)):
        assert np.array_equal(nf, targets) and nf[2] >= SW + 1


# ---------------------------------------------------------------------------------------------------------------------------
# 1e. batched voxeliser: cloud digits and the segment-length switch
# ---------------------------------------------------------------------------------------------------------------------------
def _scan_batch(small_workload, F, total=None, seed=0):
    """F small scans (slices of the workload's scans, 300 - 2000 points) with an empty scan, 1-point scans, an exact duplicate, a
    scan of repeated points, a cloud whose VoxelGrid overflows int32 and one whose keys need 31 bits (npass 4); with `total`,
    full scans are added, then the last scan is cut, so that the submission holds exactly that many points"""
    rng = np.random.default_rng(seed)
    scene = small_workload["scene"]
    base = [scene.scan(small_workload["frames"][i][2], n_beams=32, n_az=900, seed_offset=17) for i in range(6)]
    scans = []
    for i in range(F):
        b = base[i % 6]
        L = int(rng.integers(300, 2001))
        a = int(rng.integers(0, len(b) - L))
        scans.append(b[a:a + L])
    scans[3] = np.zeros((0, 4), np.float32)
    scans[5] = base[1][:1].copy()
    scans[6] = base[2][7:8].copy()
    scans[9] = scans[8].copy()
    scans[12] = np.concatenate([scans[12][:200]] * 3)
    scans[17] = np.concatenate([rng.uniform(-4.0e4, 4.0e4, (3000, 3)), rng.integers(0, 300, (3000, 1))], axis=1).astype(np.float32)
    wide = np.concatenate([rng.uniform(-250.0, 250.0, (3000, 2)), rng.uniform(-20.0, 28.0, (3000, 1)), rng.integers(0, 300, (3000, 1))], axis=1)
    wide[0, :3] = (-250.0, -250.0, -20.0)
    wide[1, :3] = (250.0, 250.0, 28.0)
    scans[F - 2] = wide.astype(np.float32)
    if total is not None:
        k = 0
        while sum(len(s) for s in scans) < total:
            j = 21 + 7 * k
            k += 1
            scans[j] = base[j % 6]
        over = sum(len(s) for s in scans) - total
        j = 21 + 7 * (k - 1)
        scans[j] = scans[j][:len(scans[j]) - over]
        assert sum(len(s) for s in scans) == total
    return scans


@pytest.mark.parametrize("F,total", [(512, None), (513, None), (1100, 2_097_152), (1100, 2_097_153)])
def test_batched_voxeliser_cloud_digits(capi, oracle_mod, small_workload, F, total):
    from test_frame_independent import oracle_query
    from test_radix_batched_model import batched_pass_plan, rs_seg_len
    p = P.preset("seq_05").replace(skip_voxelize=1)
    leaf = 0.2
    assert F <= (1 << 21) // p.num_bins                         # one node-mode submission: the batch is not split
    scans = _scan_batch(small_workload, F, total, seed=F + (total or 0))
    off = np.cumsum([0] + [len(s) for s in scans]).astype(np.uint64)
    n = int(off[-1])
    if total is not None:
        assert n == total and rs_seg_len(n) == (256 if n <= 2_097_152 else 512)
    Q = [oracle_query(oracle_mod, s, leaf, L2B) for s in scans]
    npk, ncd = batched_pass_plan(scans, leaf)
    assert npk == 4 and ncd == (1 if F <= 512 else 2)
    frames = small_workload["frames"]
    poses = np.stack([small_workload["scene"].pose7(frames[i % 6][2]) for i in range(F)]).astype(np.float64)
    m = capi.Map(small_workload["map_world"])
    h = capi.Handle(p)
    h.attach_map(m)
    keep, fk = h.process_scans(poses, np.concatenate(scans), off, leaf, L2B, want_frame_keep=True)
    stats = h.node_stats()
    xyz, qoff = h.scan_queries()
    assert len(qoff) == F + 1 and int(qoff[-1]) == sum(len(q) for q in Q)
    for f in range(F):
        got = xyz[int(qoff[f]):int(qoff[f + 1])]
        assert got.shape[0] == len(Q[f]) and np.array_equal(_bits(got), _bits(Q[f][:, :3])), f"F={F}: scan {f} query differs"
    m.reset_keep()
    keep_n, fk_n = h.process_nodes(poses, np.concatenate(Q), qoff, want_frame_keep=True)
    assert np.array_equal(fk, fk_n) and np.array_equal(keep, keep_n)
    for a, b in zip(stats, h.node_stats()):
        assert np.array_equal(a, b)
    assert (keep == 0).any()
    h.close(); m.close()
