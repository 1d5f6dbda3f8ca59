"""Crafted frames with an exact number of map points in chosen bins, for the size-threshold tests.

Every bin that `BinSpec` describes gets exactly `n` map points (ground with a chosen height distribution plus a few tall
object points, so the Scan Ratio Test flags it) and `nq` flat query points, all well inside the bin's ring / sector so that
no rounding of the binning can move a point to a neighbour.  The callers assert the counts from the oracle's own binning,
so a test cannot pass by missing the size it is about.
"""
from dataclasses import dataclass

import numpy as np

Z_KINDS = ("rough", "dup", "equal", "ulp")


@dataclass
class BinSpec:
    ring: int
    sector: int
    n: int                 # map points in the bin (ground + objects)
    z_kind: str = "rough"
    nq: int = 40           # query points in the bin
    n_obj: int = -1        # object points among the n; -1: min(60, n // 4)


def bin_id(p, ring, sector):
    return sector * p.num_rings + ring


def _inside(rng, p, ring, sector, k, lo=0.15, hi=0.85):
    """k (x, y) in the inner part [lo, hi] of the bin's ring and sector"""
    dr = p.max_range / p.num_rings
    ds = 2.0 * np.pi / p.num_sectors
    r = (ring + rng.uniform(lo, hi, k)) * dr
    th = (sector + rng.uniform(lo, hi, k)) * ds
    return r * np.cos(th), r * np.sin(th)


def ground_z(rng, kind, k):
    if kind == "dup":            # a handful of distinct heights, many exact duplicates
        return rng.choice(np.array([-1.0, -0.95, -0.9, -0.9000001, -0.0, 0.0], dtype=np.float32), k)
    if kind == "equal":          # every point at the same height
        return np.full(k, -0.9, dtype=np.float32)
    if kind == "ulp":            # clusters a few ulps wide
        return (np.float32(-0.9) + rng.integers(0, 7, k).astype(np.float32) * np.float32(6e-8)).astype(np.float32)
    assert kind == "rough"
    return rng.normal(-0.9, 0.04, k).astype(np.float32)


def bin_map_points(rng, p, s: BinSpec):
    n_obj = min(60, s.n // 4) if s.n_obj < 0 else s.n_obj
    n_g = s.n - n_obj
    gx, gy = _inside(rng, p, s.ring, s.sector, n_g)
    g = np.stack([gx, gy, ground_z(rng, s.z_kind, n_g), np.full(n_g, 40.0)], axis=1)
    ox, oy = _inside(rng, p, s.ring, s.sector, n_obj, 0.3, 0.7)
    oz = rng.uniform(-0.7, 2.0, n_obj)
    if n_obj:
        oz[0] = 2.0                                            # the bin's map height span is always > 0.5
    obj = np.stack([ox, oy, oz, np.full(n_obj, 252.0)], axis=1)
    return np.concatenate([g, obj]).astype(np.float32)


def bin_query_points(rng, p, s: BinSpec, nq=None):
    nq = s.nq if nq is None else nq
    qx, qy = _inside(rng, p, s.ring, s.sector, nq)
    qz = np.clip(rng.normal(-0.9, 0.03, nq), -0.98, -0.82)
    return np.stack([qx, qy, qz, np.full(nq, 40.0)], axis=1).astype(np.float32)


def crafted_frame(rng, p, specs, query_counts=None):
    """(map, query) with the bins of `specs`; each cloud is shuffled so a bin's points are spread over the source order.
    query_counts overrides the query points per bin (same order as specs)."""
    ms = [bin_map_points(rng, p, s) for s in specs]
    m = rng.permutation(np.concatenate(ms)) if ms else np.zeros((0, 4), np.float32)
    # the map is drawn first, so it does not depend on the query counts
    qs = [bin_query_points(rng, p, s, None if query_counts is None else query_counts[i]) for i, s in enumerate(specs)]
    q = rng.permutation(np.concatenate(qs)) if qs else np.zeros((0, 4), np.float32)
    return np.ascontiguousarray(m), np.ascontiguousarray(q)


def single_bin_frame(n, z_kind, seed, p, ring=5, sector=2):
    """One flagged bin (seq_05: ring 5, sector 2 = bin 35, about 20 m from the origin) with exactly n map points."""
    rng = np.random.default_rng(seed)
    return crafted_frame(rng, p, [BinSpec(ring, sector, n, z_kind)])
