"""An independent reference for R-GPF: a plain float64 restatement of extract_ground (erasor.cpp:233-294) against the oracle's
plane fit on the crafted single-bin frames of test_gpu_size_edges.py, at every size threshold of the CUDA kernel up to 120 000
points.  The oracle copies the reference's float arithmetic (and the CUDA kernel copies the oracle's, bit for bit), so this is the
check that the arithmetic it copies fits the right plane: normals and d within the 1e-4 bar, ground counts equal except for
points whose float64 residual lies within 1e-6 of the threshold."""
import numpy as np
import pytest

from crafted_bins import Z_KINDS, bin_id, single_bin_frame
from erasor_b200 import params as P

NORMAL_TOL = 1e-4       # north_star tolerance for plane normals / d
BORDER = 1e-6           # a float64 residual this close to the threshold may classify either way in float
SIZES = [128, 129, 256, 257, 384, 385, 512, 513, 1024, 1025, 1536, 1537, 2048, 2049, 2560, 2561, 8775, 8776, 30000, 120000]
LARGE = 8776            # above this, rough and dup ground only (as in the GPU tests)


def extract_ground_f64(pts, p):
    """float64 extract_ground of one bin's map points: [(normal, d, residual of every point)] per iteration."""
    x = pts[:, :3].astype(np.float64)
    order = np.argsort(x[:, 2], kind="stable")
    zs = x[order]
    zs = zs[np.searchsorted(zs[:, 2], p.min_h, side="left"):]          # remove_outliers: the leading z < min_h
    lw = zs[p.num_lowest_pts:p.num_lowest_pts + p.gf_num_lpr, 2]
    lpr = lw.mean() if len(lw) else 0.0
    ground = zs[zs[:, 2] < lpr + p.gf_th_seeds_height]
    out = []
    for _ in range(p.gf_iter):
        if len(ground):
            mean = ground.mean(axis=0)
            c = ground - mean
            w, v = np.linalg.eigh(c.T @ c / len(ground))
            normal = v[:, 0]
        else:
            mean, normal = np.zeros(3), np.array([0.0, 0.0, 1.0])
        d = -normal @ mean
        res = x @ normal + d
        ground = x[res < p.gf_dist_thr]
        out.append((normal, d, res))
    return out


# Findings, kept as strict expected failures so that a change in either direction shows up.
# cov_mode = 1, bin 20 m out: above 20 k seeds the float sums of PCL >= 1.11 tilt the normal by up to 8e-5 (inside the bar), and
# the 20 m lever arm turns that into |dd| of 4e-4 (30 000 points) and 1.5e-3 (120 000 points).
MISS_SHIFTED = {(30000, "dup"), (120000, "dup")}
# cov_mode = 0 (PCL <= 1.10), bin 0.6 - 3.4 m out: the unshifted float covariance misses the bar even this close to the origin,
# from 129 points on.  E[z^2] of ground at z = -0.9 is 500 times its variance, so the cancellation alone costs the normal ~1e-4;
# with near-planar ground (equal, ulp) the float normal often lands on another axis altogether (|dn| ~ 1).
MISS_UNSHIFTED = {(n, k) for n, ks in {
    129: "dup ulp", 256: "dup equal", 257: "dup ulp", 384: "rough dup equal ulp", 385: "dup equal", 512: "equal ulp",
    513: "dup equal ulp", 1024: "rough dup equal ulp", 1025: "rough dup equal ulp", 1536: "rough dup equal ulp",
    1537: "rough dup equal ulp", 2048: "rough dup equal ulp", 2049: "rough dup equal ulp", 2560: "rough dup equal ulp",
    2561: "rough dup equal ulp", 8775: "rough dup equal ulp", 8776: "rough dup equal ulp", 30000: "rough dup",
    120000: "rough dup",
}.items() for k in ks.split()}


def _cases(misses, reason):
    for n in SIZES:
        for kind in (Z_KINDS if n <= LARGE else ("rough", "dup")):
            marks = [pytest.mark.xfail(strict=True, reason=reason)] if (n, kind) in misses else []
            yield pytest.param(n, kind, marks=marks)


def _check(p, n, kind, seed, ring, sector):
    from oracle import oracle_py
    m, q = single_bin_frame(n, kind, seed, p, ring=ring, sector=sector)
    o = oracle_py.Oracle(p)
    o.run(m, q)
    b = bin_id(p, ring, sector)
    assert int(np.count_nonzero(o.bin_of_point(0) == b)) == n, "the bin must hold exactly n map points"
    planes = [x for x in o.planes() if x["bin"] == b]
    assert len(planes) == 1, "the crafted bin must be flagged"
    op = planes[0]
    assert op["n_points"] == n
    ref = extract_ground_f64(m[o.bin_of_point(0) == b], p)
    for it, (normal, d, res) in enumerate(ref):
        on, od = op["normal_d"][it, :3], op["normal_d"][it, 3]
        s = 1.0 if on @ normal >= 0 else -1.0                                # the eigenvector's sign is a convention
        err_n = np.max(np.abs(on - s * normal))
        err_d = abs(od - s * d)
        assert err_n <= NORMAL_TOL and err_d <= NORMAL_TOL, f"n={n} {kind} iteration {it}: |dn| {err_n:.2e}, |dd| {err_d:.2e}"
        r = s * res                                                          # the residual in the oracle's orientation classifies
        g64 = int(np.count_nonzero(r < p.gf_dist_thr))
        border = int(np.count_nonzero(np.abs(r - p.gf_dist_thr) <= BORDER))
        assert abs(int(op["n_ground"][it]) - g64) <= border, \
            f"n={n} {kind} iteration {it}: oracle {int(op['n_ground'][it])} ground points, float64 {g64} ({border} on the border)"
    o.close()


@pytest.mark.parametrize("n,kind", list(_cases(MISS_SHIFTED, "float sums over > 20 k seeds: d off by the 20 m lever arm")))
def test_plane_fit_shifted_covariance(n, kind):
    """cov_mode = 1 (PCL >= 1.11, shifted by the first point): the bin 20 m from the origin."""
    p = P.preset("seq_05").replace(skip_voxelize=1, version=3, cov_mode=1)
    _check(p, n, kind, seed=7000 + n, ring=5, sector=2)


@pytest.mark.parametrize("n,kind", list(_cases(MISS_UNSHIFTED, "PCL <= 1.10's unshifted float covariance")))
def test_plane_fit_unshifted_covariance_near_origin(n, kind):
    """cov_mode = 0 (PCL <= 1.10, the default) on a bin about 3 m from the origin.  Bins far from the origin are left out on
    purpose: there PCL 1.8's unshifted float covariance is dominated by rounding noise (DESIGN section 5), a property of the
    reference that the oracle and the CUDA kernel reproduce on purpose, not a fit that float64 should match."""
    p = P.preset("seq_05").replace(skip_voxelize=1, version=3, cov_mode=0)
    _check(p, n, kind, seed=9000 + n, ring=0, sector=2)
