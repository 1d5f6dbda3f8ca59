"""CPU model of the batched voxeliser's radix sort (k_node_fused<true> in erasor_b200/csrc/updater_kernels.cu): F clouds in one sort,
every cloud keyed by its own VoxelGrid, the key passes up to the largest npass of any cloud, then the cloud id as ceil(log2(NC) / 9)
more 9-bit digits (cloud_of(index) >> ((pass - npk) * 9)), and the next pass's histogram counted while scattering, as the kernel
does.  The result must be np.lexsort((index, key, cloud)): every cloud contiguous, ascending key, members in cloud order.  The
scratch carve-up of vox_plan / voxelize_tmp_bytes is restated with n_clouds (per-cloud min / max partials and first voxels)."""
import numpy as np
import pytest

from test_radix_model import K_FUSED_MAX_GRID, PART_CHUNK, RB, RD, rs_seg_len


def npass_of(n, lim):
    """vox_grid_setup: the passes a cloud of n points needs for keys < lim (an empty cloud needs none)"""
    if n == 0:
        return 0
    bits = 32
    if lim <= 0x80000000:
        bits = 1
        while (1 << bits) < lim:
            bits += 1
    return (bits + RB - 1) // RB


def cloud_digits(nc):
    cbits = int(nc - 1).bit_length() if nc > 1 else 0
    return (cbits + RB - 1) // RB


def batched_pass_plan(scans, leaf):
    """(npk, cloud digits) of one process_scans submission: VoxelGrid of every scan in float as the kernel computes it"""
    npk = 0
    inv = np.float32(1.0) / np.float32(leaf)
    for s in scans:
        if len(s) == 0:
            continue
        mn, mx = s[:, :3].min(axis=0) + np.float32(0.0), s[:, :3].max(axis=0) + np.float32(0.0)
        d = [int(np.float32(np.float32(mx[k] - mn[k]) * inv)) + 1 for k in range(3)]
        ovf = d[0] * d[1] * d[2] > 2147483647
        cells = 1
        for k in range(3):
            cells *= int(np.floor(np.float32(mx[k] * inv))) - int(np.floor(np.float32(mn[k] * inv))) + 1
        npk = max(npk, npass_of(len(s), len(s) if ovf else cells))
    return npk, cloud_digits(len(scans))


def model_batched_sort(keys, lims, off, seg):
    """(sorted keys, sorted source indices, npk, npass) by the kernel's passes; keys of cloud f are < lims[f]"""
    n = len(keys)
    NC = len(off) - 1
    nseg = (n + seg - 1) // seg
    cloud = np.searchsorted(off, np.arange(n), side="right") - 1            # cloud_of(): the first f with off[f + 1] > e
    npk = max([npass_of(int(off[f + 1] - off[f]), int(lims[f])) for f in range(NC)] + [0])
    npass = npk + cloud_digits(NC) if n else 0

    def digit(k, v, p):
        return (int(k) >> (RB * p)) & (RD - 1) if p < npk else (int(cloud[v]) >> ((p - npk) * RB)) & (RD - 1)

    k, v = keys.astype(np.uint32).copy(), np.arange(n, dtype=np.uint32)
    cnt = np.zeros((RD, nseg), dtype=np.int64)
    if n:
        np.add.at(cnt, (k & (RD - 1), np.arange(n) // seg), 1)              # pass 0 is always a key pass (npk >= 1)
    for p in range(npass):
        row_prefix = np.cumsum(cnt, axis=1) - cnt
        tot = cnt.sum(axis=1)
        base = np.cumsum(tot) - tot
        ko, vo = np.empty_like(k), np.empty_like(v)
        cnt_next = np.zeros((RD, nseg), dtype=np.int64)
        for s in range(nseg):
            nxt = base + row_prefix[:, s]
            for e in range(s * seg, min(n, (s + 1) * seg)):
                d = digit(k[e], v[e], p)
                o = nxt[d]
                nxt[d] += 1
                ko[o], vo[o] = k[e], v[e]
                if p + 1 < npass:
                    cnt_next[digit(k[e], v[e], p + 1), o // seg] += 1         # the next pass's digit, at the destination segment
        k, v, cnt = ko, vo, cnt_next
    return k, v, npk, npass


def _clouds(rng, nc, empty_every=7):
    sizes = rng.integers(0, 25, nc)
    sizes[::empty_every] = 0
    if nc > 1:
        sizes[1] = max(sizes[1], 3)
    widths = rng.choice([1, 5, 9, 10, 18, 27, 31], nc)
    lims = np.array([1 << int(w) for w in widths], dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    keys = np.empty(int(off[-1]), dtype=np.uint32)
    for f in range(nc):
        a, b = int(off[f]), int(off[f + 1])
        if b > a:
            kf = rng.integers(0, lims[f], b - a, dtype=np.int64)
            kf[rng.integers(0, b - a, (b - a) // 3)] = kf[0]                  # runs of one voxel
            kf[-1] = lims[f] - 1                                            # the cloud's key width is really needed
            keys[a:b] = kf.astype(np.uint32)
    return keys, lims, off


@pytest.mark.parametrize("nc", [1, 2, 511, 512, 513, 1000])
def test_batched_sort_is_the_lexsort(nc):
    rng = np.random.default_rng(nc)
    keys, lims, off = _clouds(rng, nc)
    if nc > 1:                                                              # one cloud with 31-bit keys: npk = 4
        a, b = int(off[1]), int(off[2])
        lims[1] = 1 << 31
        keys[a:b] = rng.integers(0, 1 << 31, b - a, dtype=np.int64).astype(np.uint32)
        keys[b - 1] = (1 << 31) - 1
    k, v, npk, npass = model_batched_sort(keys, lims, off, 256)
    cloud = np.searchsorted(off, np.arange(len(keys)), side="right") - 1
    order = np.lexsort((np.arange(len(keys)), keys, cloud))
    assert np.array_equal(v, order.astype(np.uint32)) and np.array_equal(k, keys[order])
    assert npass == npk + cloud_digits(nc)
    if nc > 1:
        assert npk == 4
    assert cloud_digits(nc) == (0 if nc == 1 else 1 if nc <= 512 else 2)


def test_scratch_carve_up_with_clouds():
    for n in (0, 1, 255, 256, 110_000, 2_097_152, 2_097_153, 50_000_000):
        for nc in (1, 2, 512, 513, 2330):
            seg = rs_seg_len(n)
            nseg = (n + seg - 1) // seg
            # vox_plan(tmp, n, n_clouds): key / idx ping-pong, two histogram matrices RD x (nseg + 1), digit totals, head-chunk
            # counters, voxel starts / keys, per-cloud min / max partials (6 per CTA), first voxel of every cloud
            used = 4 * n + 2 * RD * (nseg + 1) + RD + ((n + PART_CHUNK - 1) // PART_CHUNK + 1) + 2 * (n + 2) + 6 * K_FUSED_MAX_GRID * nc + nc
            # voxelize_tmp_bytes(n, n_clouds) in words
            have = (4 * n + 2 * RD * ((n + seg - 1) // seg + 1) + RD + ((n + PART_CHUNK - 1) // PART_CHUNK + 1) + 2 * (n + 2) + 64
                    + 6 * K_FUSED_MAX_GRID * nc + nc)
            assert used <= have, (n, nc)
