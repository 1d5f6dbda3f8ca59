"""ctypes binding of the C ABI in ``include/erasor_b200.h`` (``erasor_b200/_lib/liberasor_b200.so``).

The library is CUDA-only: importing this module without the built ``.so`` raises, and
``Handle(...)`` raises when there is no CUDA device.  There is no CPU fallback anywhere in the
package (the CPU oracle lives under ``oracle/`` and is test infrastructure).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_size_t, c_uint8, c_uint32, c_uint64, c_void_p

import numpy as np

from .params import ErasorParams, ErasorParamsC

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liberasor_b200.so")

PTR_HOST, PTR_DEVICE = 0, 1
PTR_QUERY_XYZ = 16          # OR-able (mask modes): the query cloud is packed x y z, three floats per point
CLOUD_MAP, CLOUD_QUERY = 0, 1
OK, E_INVALID, E_CUDA, E_STATE, E_CAPACITY, E_UNSUPPORTED = 0, -1, -2, -3, -4, -5

EXPORTS = [
    "erasor_create", "erasor_destroy", "erasor_last_error", "erasor_abi_version", "erasor_stream", "erasor_synchronize",
    "erasor_set_inputs", "erasor_compare", "erasor_get_output_sizes", "erasor_get_static_estimate", "erasor_get_outliers",
    "erasor_get_max_range", "erasor_device_outputs", "erasor_get_ground_viz", "erasor_get_bins", "erasor_get_status", "erasor_get_planes", "erasor_get_static_mask",
    "erasor_get_fence_counts", "erasor_process_frames", "erasor_process_frames_async", "erasor_wait", "erasor_process_frames_fold",
    "erasor_process_frames_fold_async", "erasor_fold_keep_masks", "erasor_reset_keep_mask", "erasor_get_frame_stats", "erasor_kernel_launch_count",
    "erasor_map_create", "erasor_map_destroy", "erasor_map_size", "erasor_map_reset_keep", "erasor_map_get_keep", "erasor_map_keep_device",
    "erasor_map_points_device", "erasor_attach_map", "erasor_process_nodes", "erasor_process_nodes_async", "erasor_get_node_stats",
    "erasor_comm_unique_id", "erasor_comm_init", "erasor_comm_destroy", "erasor_allgather_and_keep", "erasor_and_keep_masks",
    "erasor_get_kernel_time_ms", "erasor_reset_kernel_times", "erasor_get_rgpf_profile", "erasor_get_srt_profile",
    "erasor_process_scans", "erasor_process_scans_async", "erasor_get_scan_queries", "erasor_save_static_map",
    "erasor_updater_create", "erasor_updater_destroy", "erasor_updater_reset", "erasor_updater_last_error", "erasor_updater_process_node", "erasor_updater_prefetch_scan",
    "erasor_updater_map_size", "erasor_updater_get_cloud", "erasor_updater_save_static_map", "erasor_updater_voxelize", "erasor_updater_mapgen_node",
    "erasor_updater_erasor", "erasor_updater_kernel_launch_count", "erasor_updater_get_fused_profile",
]


class UpdaterParamsC(ctypes.Structure):
    """erasor_updater_params_t"""
    _fields_ = [
        ("query_voxel_size", c_double), ("map_voxel_size", c_double), ("removal_interval", c_int), ("is_large_scale", c_int),
        ("submap_size", c_double), ("max_range", c_double), ("version", c_int), ("pad_", c_int), ("lidar2body", c_double * 7),
    ]


class ScanParamsC(ctypes.Structure):
    """erasor_scan_params_t"""
    _fields_ = [("query_voxel_size", c_double), ("lidar2body", c_double * 7)]


def scan_params(query_voxel_size: float, lidar2body) -> ScanParamsC:
    sp = ScanParamsC()
    sp.query_voxel_size = float(query_voxel_size)
    l2b = np.asarray(lidar2body, dtype=np.float64).reshape(7)
    for i in range(7):
        sp.lidar2body[i] = float(l2b[i])
    return sp


class ErasorError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"erasor_b200 error {code}: {msg}")
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with erasor_b200/csrc/build.sh (or __graft_entry__.build()). "
            "erasor_b200 has no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    fp = POINTER(c_float)
    L.erasor_create.restype = c_int
    L.erasor_create.argtypes = [POINTER(ErasorParamsC), c_int, POINTER(c_void_p)]
    L.erasor_destroy.restype = None
    L.erasor_destroy.argtypes = [c_void_p]
    L.erasor_last_error.restype = c_char_p
    L.erasor_last_error.argtypes = [c_void_p]
    L.erasor_abi_version.restype = c_int
    L.erasor_stream.restype = c_void_p
    L.erasor_stream.argtypes = [c_void_p]
    L.erasor_synchronize.argtypes = [c_void_p]
    L.erasor_set_inputs.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, c_int]
    L.erasor_compare.argtypes = [c_void_p, c_int, c_int]
    L.erasor_get_output_sizes.argtypes = [c_void_p, POINTER(c_size_t), POINTER(c_size_t), POINTER(c_size_t), POINTER(c_size_t)]
    L.erasor_get_static_estimate.argtypes = [c_void_p, c_void_p, c_size_t, POINTER(c_size_t), c_void_p, c_size_t, POINTER(c_size_t), c_int]
    L.erasor_get_outliers.argtypes = [c_void_p, c_void_p, c_size_t, POINTER(c_size_t), c_void_p, c_size_t, POINTER(c_size_t), c_int]
    L.erasor_get_ground_viz.argtypes = [c_void_p, c_void_p, c_size_t, POINTER(c_size_t), c_int]
    L.erasor_get_max_range.restype = c_double
    L.erasor_get_max_range.argtypes = [c_void_p]
    L.erasor_get_bins.argtypes = [c_void_p, c_int, POINTER(c_int32), fp, fp, POINTER(c_uint32)]
    L.erasor_get_status.argtypes = [c_void_p, fp]
    L.erasor_get_planes.argtypes = [c_void_p, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), POINTER(c_double),
                                    POINTER(c_double), POINTER(c_int32), POINTER(c_size_t)]
    L.erasor_get_static_mask.argtypes = [c_void_p, POINTER(c_uint8), POINTER(c_uint8)]
    L.erasor_get_fence_counts.argtypes = [c_void_p, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint64)]
    L.erasor_process_frames.argtypes = [c_void_p, c_void_p, POINTER(c_uint64), c_void_p, POINTER(c_uint64), c_int, c_void_p, c_int]
    L.erasor_process_frames_fold.argtypes = [c_void_p, c_void_p, POINTER(c_uint64), c_void_p, POINTER(c_uint64), c_int, c_void_p, c_int,
                                             c_void_p, c_void_p, c_size_t]
    L.erasor_fold_keep_masks.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_size_t]
    L.erasor_process_frames_async.argtypes = L.erasor_process_frames.argtypes
    L.erasor_process_frames_fold_async.argtypes = L.erasor_process_frames_fold.argtypes
    L.erasor_wait.argtypes = [c_void_p]
    L.erasor_reset_keep_mask.argtypes = [c_void_p, c_void_p, c_size_t]
    L.erasor_map_create.argtypes = [c_void_p, c_size_t, c_int, c_int, POINTER(c_void_p)]
    L.erasor_map_destroy.restype = None
    L.erasor_map_destroy.argtypes = [c_void_p]
    L.erasor_map_size.restype = c_size_t
    L.erasor_map_size.argtypes = [c_void_p]
    L.erasor_map_reset_keep.argtypes = [c_void_p]
    L.erasor_map_get_keep.argtypes = [c_void_p, c_void_p, c_int]
    L.erasor_map_keep_device.restype = c_void_p
    L.erasor_map_keep_device.argtypes = [c_void_p]
    L.erasor_map_points_device.restype = c_void_p
    L.erasor_map_points_device.argtypes = [c_void_p]
    L.erasor_attach_map.argtypes = [c_void_p, c_void_p]
    L.erasor_process_nodes.argtypes = [c_void_p, POINTER(c_double), c_void_p, POINTER(c_uint64), c_int, c_double, c_void_p, c_void_p, c_int]
    L.erasor_process_nodes_async.argtypes = L.erasor_process_nodes.argtypes
    L.erasor_get_node_stats.argtypes = [c_void_p, POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32)]
    L.erasor_process_scans.argtypes = [c_void_p, POINTER(ScanParamsC), POINTER(c_double), c_void_p, POINTER(c_uint64), c_int, c_double, c_void_p,
                                       c_void_p, c_int]
    L.erasor_process_scans_async.argtypes = L.erasor_process_scans.argtypes
    L.erasor_get_scan_queries.argtypes = [c_void_p, c_void_p, c_size_t, POINTER(c_uint64)]
    L.erasor_save_static_map.argtypes = [c_void_p, c_float, c_void_p, c_size_t, POINTER(c_size_t)]
    L.erasor_comm_unique_id.argtypes = [c_void_p]
    L.erasor_comm_init.argtypes = [c_void_p, c_void_p, c_int, c_int]
    L.erasor_comm_destroy.argtypes = [c_void_p]
    L.erasor_allgather_and_keep.argtypes = [c_void_p, c_void_p, c_size_t]
    L.erasor_and_keep_masks.argtypes = [c_void_p, c_void_p, c_int, c_size_t, c_void_p]
    L.erasor_get_frame_stats.argtypes = [c_void_p, POINTER(c_uint32), POINTER(c_uint32)]
    L.erasor_kernel_launch_count.restype = c_uint64
    L.erasor_kernel_launch_count.argtypes = [c_void_p]
    L.erasor_get_kernel_time_ms.argtypes = [c_void_p, c_int, POINTER(c_double), POINTER(c_uint64)]
    L.erasor_reset_kernel_times.argtypes = [c_void_p, c_int]
    L.erasor_get_rgpf_profile.argtypes = [c_void_p, POINTER(c_uint32), POINTER(c_uint32), POINTER(c_size_t)]
    L.erasor_get_srt_profile.argtypes = [c_void_p, POINTER(c_uint32)]
    L.erasor_updater_create.argtypes = [POINTER(UpdaterParamsC), POINTER(ErasorParamsC), c_void_p, c_size_t, c_int, POINTER(c_void_p)]
    L.erasor_updater_destroy.restype = None
    L.erasor_updater_destroy.argtypes = [c_void_p]
    L.erasor_updater_reset.argtypes = [c_void_p, c_void_p, c_size_t]
    L.erasor_updater_last_error.restype = c_char_p
    L.erasor_updater_last_error.argtypes = [c_void_p]
    L.erasor_updater_process_node.argtypes = [c_void_p, c_int, POINTER(c_double), c_void_p, c_size_t, c_int, POINTER(c_int)]
    L.erasor_updater_prefetch_scan.argtypes = [c_void_p, c_void_p, c_size_t, c_int]
    L.erasor_updater_map_size.argtypes = [c_void_p, POINTER(c_size_t)]
    L.erasor_updater_get_cloud.argtypes = [c_void_p, c_int, c_void_p, c_size_t, POINTER(c_size_t), c_int]
    L.erasor_updater_save_static_map.argtypes = [c_void_p, c_float, c_void_p, c_size_t, POINTER(c_size_t)]
    L.erasor_updater_voxelize.argtypes = [c_void_p, c_void_p, c_size_t, c_float, c_void_p, c_size_t, POINTER(c_size_t)]
    L.erasor_updater_mapgen_node.argtypes = [c_void_p, POINTER(c_double), c_void_p, c_size_t, c_int, c_void_p, c_size_t, POINTER(c_size_t)]
    L.erasor_updater_erasor.restype = c_void_p
    L.erasor_updater_erasor.argtypes = [c_void_p]
    L.erasor_updater_kernel_launch_count.restype = c_uint64
    L.erasor_updater_kernel_launch_count.argtypes = [c_void_p]
    L.erasor_updater_get_fused_profile.argtypes = [c_void_p, c_void_p]
    return L


_L = None


def lib():
    global _L
    if _L is None:
        _L = _load()
    return _L


def _cloud(a) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.size == 0:
        return a.reshape(0, 4)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError("clouds are float32 [n,4] = x,y,z,intensity")
    return a


class Handle:
    """One ``erasor_handle_t``: one CUDA device, one stream, fixed parameters."""

    def __init__(self, params: ErasorParams, device: int = 0):
        self.L = lib()
        self.params = params
        self._pc = params.to_c()
        h = c_void_p()
        rc = self.L.erasor_create(ctypes.byref(self._pc), device, ctypes.byref(h))
        if rc != OK:
            raise ErasorError(rc, (self.L.erasor_last_error(None) or b"").decode())
        self.h = h
        self.n_map = 0
        self.n_query = 0
        self._keep = []   # keeps host arrays alive while the library may still read them

    # -- plumbing ---------------------------------------------------------------------------
    def _ck(self, rc: int):
        if rc != OK:
            raise ErasorError(rc, (self.L.erasor_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.erasor_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def stream(self) -> int:
        return self.L.erasor_stream(self.h) or 0

    def synchronize(self):
        self._ck(self.L.erasor_synchronize(self.h))

    # -- the per-frame path ---------------------------------------------------------------
    def set_inputs(self, map_voi, query_voi):
        m, q = _cloud(map_voi), _cloud(query_voi)
        self._keep = [m, q]
        self.n_map, self.n_query = len(m), len(q)
        self._ck(self.L.erasor_set_inputs(self.h, m.ctypes.data, len(m), q.ctypes.data, len(q), PTR_HOST))

    def set_inputs_device(self, map_ptr: int, n_map: int, query_ptr: int, n_query: int):
        self.n_map, self.n_query = n_map, n_query
        self._ck(self.L.erasor_set_inputs(self.h, c_void_p(map_ptr), n_map, c_void_p(query_ptr), n_query, PTR_DEVICE))

    def compare(self, version: int | None = None, frame: int = 0):
        self._ck(self.L.erasor_compare(self.h, self.params.version if version is None else version, frame))

    def output_sizes(self):
        a, c, m, q = c_size_t(), c_size_t(), c_size_t(), c_size_t()
        self._ck(self.L.erasor_get_output_sizes(self.h, ctypes.byref(a), ctypes.byref(c), ctypes.byref(m), ctypes.byref(q)))
        return a.value, c.value, m.value, q.value

    def get_static_estimate(self):
        na, nc, _, _ = self.output_sizes()
        arr = np.empty((na, 4), dtype=np.float32)
        cmp_ = np.empty((nc, 4), dtype=np.float32)
        a, c = c_size_t(), c_size_t()
        self._ck(self.L.erasor_get_static_estimate(self.h, arr.ctypes.data, na, ctypes.byref(a), cmp_.ctypes.data, nc, ctypes.byref(c), PTR_HOST))
        return arr, cmp_

    def get_outliers(self):
        _, _, nm, nq = self.output_sizes()
        mr = np.empty((nm, 4), dtype=np.float32)
        cr = np.empty((nq, 4), dtype=np.float32)
        a, c = c_size_t(), c_size_t()
        self._ck(self.L.erasor_get_outliers(self.h, mr.ctypes.data, nm, ctypes.byref(a), cr.ctypes.data, nq, ctypes.byref(c), PTR_HOST))
        return mr, cr

    def get_ground_viz(self) -> np.ndarray:
        n = c_size_t(0)
        self._ck(self.L.erasor_get_ground_viz(self.h, None, 0, ctypes.byref(n), PTR_HOST))
        out = np.empty((n.value, 4), dtype=np.float32)
        if n.value:
            self._ck(self.L.erasor_get_ground_viz(self.h, out.ctypes.data, n.value, ctypes.byref(n), PTR_HOST))
        return out

    def get_max_range(self) -> float:
        return self.L.erasor_get_max_range(self.h)

    # -- parity taps ---------------------------------------------------------------------------
    def get_bins(self, which: int):
        B = self.params.num_bins
        n = self.n_map if which == CLOUD_MAP else self.n_query
        bop = np.empty(n, dtype=np.int32)
        mn, mx = np.empty(B, dtype=np.float32), np.empty(B, dtype=np.float32)
        cnt = np.empty(B, dtype=np.uint32)
        self._ck(self.L.erasor_get_bins(self.h, which, bop.ctypes.data_as(POINTER(c_int32)), mn.ctypes.data_as(POINTER(c_float)),
                                        mx.ctypes.data_as(POINTER(c_float)), cnt.ctypes.data_as(POINTER(c_uint32))))
        return bop, mn, mx, cnt

    def get_status(self) -> np.ndarray:
        st = np.empty(self.params.num_bins, dtype=np.float32)
        self._ck(self.L.erasor_get_status(self.h, st.ctypes.data_as(POINTER(c_float))))
        return st

    def get_planes(self):
        n = c_size_t(0)
        self._ck(self.L.erasor_get_planes(self.h, None, None, None, None, None, None, ctypes.byref(n)))
        k, it = n.value, self.params.gf_iter
        bins, npts, nseeds = (np.zeros(k, dtype=np.int32) for _ in range(3))
        lpr = np.zeros(k)
        nd = np.zeros((k, it, 4))
        ng = np.zeros((k, it), dtype=np.int32)
        cap = c_size_t(k)
        if k:
            self._ck(self.L.erasor_get_planes(self.h, bins.ctypes.data_as(POINTER(c_int32)), npts.ctypes.data_as(POINTER(c_int32)),
                                              nseeds.ctypes.data_as(POINTER(c_int32)), lpr.ctypes.data_as(POINTER(c_double)),
                                              nd.ctypes.data_as(POINTER(c_double)), ng.ctypes.data_as(POINTER(c_int32)), ctypes.byref(cap)))
        return [dict(bin=int(bins[i]), n_points=int(npts[i]), n_seeds=int(nseeds[i]), lpr=float(lpr[i]), normal_d=nd[i], n_ground=ng[i])
                for i in range(k)]

    def get_static_mask(self):
        keep = np.empty(self.n_map, dtype=np.uint8)
        gnd = np.empty(self.n_map, dtype=np.uint8)
        self._ck(self.L.erasor_get_static_mask(self.h, keep.ctypes.data_as(POINTER(c_uint8)), gnd.ctypes.data_as(POINTER(c_uint8))))
        return keep, gnd

    def fence_counts(self):
        a, b, c = c_uint64(), c_uint64(), c_uint64()
        self._ck(self.L.erasor_get_fence_counts(self.h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return dict(negzero_points=a.value, empty_plane_fits=b.value, ambiguous_sector=c.value)

    # -- batch mode ---------------------------------------------------------------------------
    def process_frames(self, map_xyzi, map_offsets, query_xyzi, query_offsets) -> np.ndarray:
        """Host-buffer batch call: returns keep mask (uint8) over all map points of all frames."""
        m, q = _cloud(map_xyzi), _cloud(query_xyzi)
        mo = np.ascontiguousarray(map_offsets, dtype=np.uint64)
        qo = np.ascontiguousarray(query_offsets, dtype=np.uint64)
        F = len(mo) - 1
        keep = np.empty(int(mo[-1]), dtype=np.uint8)
        self._ck(self.L.erasor_process_frames(self.h, m.ctypes.data, mo.ctypes.data_as(POINTER(c_uint64)), q.ctypes.data,
                                              qo.ctypes.data_as(POINTER(c_uint64)), F, keep.ctypes.data, PTR_HOST))
        self.n_frames = F
        return keep

    def process_frames_ptr(self, map_ptr: int, map_offsets: np.ndarray, query_ptr: int, query_offsets: np.ndarray, keep_ptr: int, ptr_kind: int,
                           fold=None, asynchronous: bool = False):
        """Raw-pointer batch call (device tensors or pinned host memory); offsets are host uint64 arrays.
        The ctypes views of the offset arrays are cached per array object so that a caller streaming equally-shaped
        batches pays one foreign call per step and nothing else."""
        key = (id(map_offsets), id(query_offsets))
        c = getattr(self, "_off_cache", None)
        if c is None or c[0] != key:
            mo = np.ascontiguousarray(map_offsets, dtype=np.uint64)
            qo = np.ascontiguousarray(query_offsets, dtype=np.uint64)
            c = (key, mo, qo, mo.ctypes.data_as(POINTER(c_uint64)), qo.ctypes.data_as(POINTER(c_uint64)), len(mo) - 1)
            self._off_cache = c
        if fold is None:
            fn = self.L.erasor_process_frames_async if asynchronous else self.L.erasor_process_frames
            rc = fn(self.h, map_ptr, c[3], query_ptr, c[4], c[5], keep_ptr, ptr_kind)
        else:       # fold = (voi_index device ptr, global_keep device ptr, n_global): the fold runs in R-GPF's epilogue
            fn = self.L.erasor_process_frames_fold_async if asynchronous else self.L.erasor_process_frames_fold
            rc = fn(self.h, map_ptr, c[3], query_ptr, c[4], c[5], keep_ptr, ptr_kind, fold[0], fold[1], fold[2])
        if rc != OK:
            self._ck(rc)
        self.n_frames = c[5]

    def fold_keep_masks(self, keep_ptr: int, voi_index_ptr: int, n: int, global_keep_ptr: int, n_global: int):
        """device pointers; asynchronous on the handle's stream; accumulates (reset_keep_mask starts a job)"""
        self._ck(self.L.erasor_fold_keep_masks(self.h, c_void_p(keep_ptr), c_void_p(voi_index_ptr), n, c_void_p(global_keep_ptr), n_global))

    def reset_keep_mask(self, global_keep_ptr: int, n_global: int):
        self._ck(self.L.erasor_reset_keep_mask(self.h, c_void_p(global_keep_ptr), n_global))

    def wait(self):
        """Complete the handle's asynchronous submission (``*_async``)."""
        rc = self.L.erasor_wait(self.h)
        if rc != OK:
            self._ck(rc)

    # -- map-resident node mode -----------------------------------------------------------------
    def attach_map(self, m: "Map"):
        self._ck(self.L.erasor_attach_map(self.h, m.h if m is not None else None))
        self._map = m

    def process_nodes(self, poses7, query_xyzi, query_offsets, voi_max_range: float = 0.0, want_frame_keep: bool = False, packed_xyz: bool = False):
        """Host-buffer node batch: returns (folded keep mask of the map after this batch, per-frame masks or None).
        packed_xyz: ship the queries as packed x y z (ERASOR_PTR_QUERY_XYZ) -- the masks do not depend on the intensity."""
        P = np.ascontiguousarray(poses7, dtype=np.float64).reshape(-1, 7)
        q = _cloud(query_xyzi)
        if packed_xyz:
            q = np.ascontiguousarray(q[:, :3])
        qo = np.ascontiguousarray(query_offsets, dtype=np.uint64)
        F = len(qo) - 1
        assert len(P) == F
        n = self._map.size
        keep = np.empty(n, dtype=np.uint8)
        fk = np.empty((F, n), dtype=np.uint8) if want_frame_keep else None
        self._ck(self.L.erasor_process_nodes(self.h, P.ctypes.data_as(POINTER(c_double)), q.ctypes.data, qo.ctypes.data_as(POINTER(c_uint64)), F,
                                             float(voi_max_range), fk.ctypes.data if fk is not None else None, keep.ctypes.data,
                                             PTR_HOST | (PTR_QUERY_XYZ if packed_xyz else 0)))
        self.n_frames = F
        return keep, fk

    def process_nodes_ptr(self, poses7: np.ndarray, query_ptr: int, query_offsets: np.ndarray, voi_max_range: float, frame_keep_ptr: int,
                          keep_out_ptr: int, ptr_kind: int, asynchronous: bool = False):
        """Raw-pointer node batch (device tensors or pinned host memory).  poses7: contiguous float64 [F,7]; offsets uint64 [F+1]."""
        key = (id(poses7), id(query_offsets))
        c = getattr(self, "_node_cache", None)
        if c is None or c[0] != key:
            assert poses7.dtype == np.float64 and poses7.flags["C_CONTIGUOUS"] and query_offsets.dtype == np.uint64
            c = (key, poses7, query_offsets, poses7.ctypes.data_as(POINTER(c_double)), query_offsets.ctypes.data_as(POINTER(c_uint64)), len(query_offsets) - 1)
            self._node_cache = c
        fn = self.L.erasor_process_nodes_async if asynchronous else self.L.erasor_process_nodes
        rc = fn(self.h, c[3], query_ptr, c[4], c[5], voi_max_range, frame_keep_ptr or None, keep_out_ptr or None, ptr_kind)
        if rc != OK:
            self._ck(rc)
        self.n_frames = c[5]

    def process_scans(self, poses7, scans, scan_offsets, query_voxel_size: float, lidar2body, voi_max_range: float = 0.0,
                      want_frame_keep: bool = False, packed_xyz: bool = False):
        """Node batch on raw LiDAR-frame scans (erasor_process_scans): each scan is voxelised at query_voxel_size and moved to the
        body frame by lidar2body (x y z qx qy qz qw) on the device, then processed as process_nodes does.  scans: float32 [n,4]
        (x y z i) or [n,3]; packed_xyz ships them as 12 bytes per point.  Returns (folded keep mask, per-frame masks or None)."""
        P = np.ascontiguousarray(poses7, dtype=np.float64).reshape(-1, 7)
        q = np.ascontiguousarray(scans, dtype=np.float32)
        if q.size == 0:
            q = q.reshape(0, 4)
        if q.ndim != 2 or q.shape[1] not in (3, 4):
            raise ValueError("scans are float32 [n,4] (x y z i) or [n,3] (x y z)")
        if packed_xyz and q.shape[1] == 4:
            q = np.ascontiguousarray(q[:, :3])
        if not packed_xyz and q.shape[1] == 3:
            raise ValueError("[n,3] scans need packed_xyz=True")
        so = np.ascontiguousarray(scan_offsets, dtype=np.uint64)
        F = len(so) - 1
        assert len(P) == F
        n = self._map.size
        keep = np.empty(n, dtype=np.uint8)
        fk = np.empty((F, n), dtype=np.uint8) if want_frame_keep else None
        sp = scan_params(query_voxel_size, lidar2body)
        self._ck(self.L.erasor_process_scans(self.h, ctypes.byref(sp), P.ctypes.data_as(POINTER(c_double)), q.ctypes.data if q.size else None,
                                             so.ctypes.data_as(POINTER(c_uint64)), F, float(voi_max_range),
                                             fk.ctypes.data if fk is not None else None, keep.ctypes.data,
                                             PTR_HOST | (PTR_QUERY_XYZ if packed_xyz else 0)))
        self.n_frames = F
        return keep, fk

    def process_scans_ptr(self, sp: ScanParamsC, poses7: np.ndarray, scans_ptr: int, scan_offsets: np.ndarray, voi_max_range: float,
                          frame_keep_ptr: int, keep_out_ptr: int, ptr_kind: int, asynchronous: bool = False):
        """Raw-pointer form of process_scans (device tensors or pinned host memory; ptr_kind may carry PTR_QUERY_XYZ).
        sp: scan_params(...); poses7: contiguous float64 [F,7]; offsets uint64 [F+1]."""
        assert poses7.dtype == np.float64 and poses7.flags["C_CONTIGUOUS"] and scan_offsets.dtype == np.uint64
        F = len(scan_offsets) - 1
        fn = self.L.erasor_process_scans_async if asynchronous else self.L.erasor_process_scans
        rc = fn(self.h, ctypes.byref(sp), poses7.ctypes.data_as(POINTER(c_double)), scans_ptr or None, scan_offsets.ctypes.data_as(POINTER(c_uint64)),
                F, float(voi_max_range), frame_keep_ptr or None, keep_out_ptr or None, ptr_kind)
        if rc != OK:
            self._ck(rc)
        self.n_frames = F

    def scan_queries(self):
        """The voxelised body-frame queries of the last process_scans submission: (x y z float32 [n,3], offsets uint64 [F+1])."""
        F = self.n_frames
        off = np.zeros(F + 1, dtype=np.uint64)
        self._ck(self.L.erasor_get_scan_queries(self.h, None, 0, off.ctypes.data_as(POINTER(c_uint64))))
        xyz = np.empty((max(int(off[-1]), 1), 3), dtype=np.float32)
        self._ck(self.L.erasor_get_scan_queries(self.h, xyz.ctypes.data, len(xyz), off.ctypes.data_as(POINTER(c_uint64))))
        return xyz[:int(off[-1])].copy(), off

    def save_static_map(self, voxel_size: float) -> np.ndarray:
        """save_static_map of the attached map: voxelize_preserving_labels(map[keep == 1], voxel_size), float32 [n,4]."""
        n = c_size_t(0)
        self._ck(self.L.erasor_save_static_map(self.h, float(voxel_size), None, 0, ctypes.byref(n)))
        out = np.empty((max(n.value, 1), 4), dtype=np.float32)
        self._ck(self.L.erasor_save_static_map(self.h, float(voxel_size), out.ctypes.data, len(out), ctypes.byref(n)))
        return out[:n.value].copy()

    def node_stats(self):
        F = self.n_frames
        nv, nf, nr = (np.zeros(F, dtype=np.uint32) for _ in range(3))
        self._ck(self.L.erasor_get_node_stats(self.h, nv.ctypes.data_as(POINTER(c_uint32)), nf.ctypes.data_as(POINTER(c_uint32)),
                                              nr.ctypes.data_as(POINTER(c_uint32))))
        return nv, nf, nr

    # -- the exchange step ------------------------------------------------------------------------
    def comm_init(self, id128: bytes, n_ranks: int, rank: int):
        buf = (ctypes.c_uint8 * 128).from_buffer_copy(id128)
        self._ck(self.L.erasor_comm_init(self.h, buf, n_ranks, rank))

    def comm_destroy(self):
        self._ck(self.L.erasor_comm_destroy(self.h))

    def and_keep_masks(self, masks_ptr: int, n_masks: int, n: int, out_ptr: int):
        self._ck(self.L.erasor_and_keep_masks(self.h, c_void_p(masks_ptr), n_masks, n, c_void_p(out_ptr)))

    def allgather_and_keep(self, global_keep_ptr: int, n_global: int):
        """device pointer; asynchronous on the handle's stream; no-op without a communicator"""
        self._ck(self.L.erasor_allgather_and_keep(self.h, c_void_p(global_keep_ptr), n_global))

    def frame_stats(self):
        F = self.n_frames
        nf, nr = np.zeros(F, dtype=np.uint32), np.zeros(F, dtype=np.uint32)
        self._ck(self.L.erasor_get_frame_stats(self.h, nf.ctypes.data_as(POINTER(c_uint32)), nr.ctypes.data_as(POINTER(c_uint32))))
        return nf, nr

    # -- instrumentation ------------------------------------------------------------------------
    def kernel_launch_count(self) -> int:
        return int(self.L.erasor_kernel_launch_count(self.h))

    def reset_kernel_times(self, enable: bool):
        self._ck(self.L.erasor_reset_kernel_times(self.h, 1 if enable else 0))

    def srt_profile(self):
        out = np.zeros(8, dtype=np.uint32)
        self._ck(self.L.erasor_get_srt_profile(self.h, out.ctypes.data_as(POINTER(c_uint32))))
        return out

    def rgpf_profile(self):
        n = c_size_t(0)
        self._ck(self.L.erasor_get_rgpf_profile(self.h, None, None, ctypes.byref(n)))
        k = n.value
        npts = np.zeros(k, dtype=np.uint32)
        prof = np.zeros((k, 8), dtype=np.uint32)
        cap = c_size_t(k)
        if k:
            self._ck(self.L.erasor_get_rgpf_profile(self.h, npts.ctypes.data_as(POINTER(c_uint32)), prof.ctypes.data_as(POINTER(c_uint32)), ctypes.byref(cap)))
        return npts, prof

    def kernel_time_ms(self, kernel_id: int):
        t, n = c_double(), c_uint64()
        self._ck(self.L.erasor_get_kernel_time_ms(self.h, kernel_id, ctypes.byref(t), ctypes.byref(n)))
        return t.value, n.value


def comm_unique_id() -> bytes:
    """NCCL unique id for erasor_comm_init (call on rank 0, ship the bytes to the other ranks)."""
    buf = (ctypes.c_uint8 * 128)()
    rc = lib().erasor_comm_unique_id(buf)
    if rc != OK:
        raise ErasorError(rc, (lib().erasor_last_error(None) or b"").decode())
    return bytes(buf)


class Map:
    """One ``erasor_map_t``: the global map resident in HBM plus its global keep mask."""

    def __init__(self, map_xyzi=None, device: int = 0, device_ptr: int = 0, n: int = 0):
        self.L = lib()
        h = c_void_p()
        if device_ptr:
            rc = self.L.erasor_map_create(c_void_p(device_ptr), n, PTR_DEVICE, device, ctypes.byref(h))
        else:
            m = _cloud(map_xyzi)
            rc = self.L.erasor_map_create(m.ctypes.data, len(m), PTR_HOST, device, ctypes.byref(h))
        if rc != OK:
            raise ErasorError(rc, (self.L.erasor_last_error(None) or b"").decode())
        self.h = h

    @property
    def size(self) -> int:
        return int(self.L.erasor_map_size(self.h))

    @property
    def keep_ptr(self) -> int:
        return self.L.erasor_map_keep_device(self.h) or 0

    def reset_keep(self):
        rc = self.L.erasor_map_reset_keep(self.h)
        if rc != OK:
            raise ErasorError(rc, "erasor_map_reset_keep")

    def get_keep(self) -> np.ndarray:
        out = np.empty(self.size, dtype=np.uint8)
        rc = self.L.erasor_map_get_keep(self.h, out.ctypes.data, PTR_HOST)
        if rc != OK:
            raise ErasorError(rc, "erasor_map_get_keep")
        return out

    def close(self):
        if getattr(self, "h", None):
            self.L.erasor_map_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Updater:
    """Device-resident mirror of ``erasor::OfflineMapUpdater`` (one ``erasor_updater_t``)."""
    MAP_ARRANGED, MAP_VOI, QUERY_VOI, MAP_REJECTED, OUTSKIRTS, SUBMAP_COMPLEMENT = 0, 1, 2, 5, 7, 8

    def __init__(self, up, ep: ErasorParams, initial_map, device: int = 0):
        self.L = lib()
        self.ep, self.up = ep, up
        upc = UpdaterParamsC()
        upc.query_voxel_size, upc.map_voxel_size = up.query_voxel_size, up.map_voxel_size
        upc.removal_interval, upc.is_large_scale = up.removal_interval, 1 if up.is_large_scale else 0
        upc.submap_size, upc.max_range, upc.version = up.submap_size, up.max_range, up.version
        for i in range(7):
            upc.lidar2body[i] = up.lidar2body[i]
        self._upc, self._epc = upc, ep.to_c()
        m = _cloud(initial_map)
        h = c_void_p()
        rc = self.L.erasor_updater_create(ctypes.byref(upc), ctypes.byref(self._epc), m.ctypes.data, len(m), device, ctypes.byref(h))
        if rc != OK:
            raise ErasorError(rc, (self.L.erasor_updater_last_error(None) or b"").decode())
        self.h = h

    def _ck(self, rc: int):
        if rc != OK:
            raise ErasorError(rc, (self.L.erasor_updater_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.erasor_updater_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, initial_map):
        m = _cloud(initial_map)
        self._ck(self.L.erasor_updater_reset(self.h, m.ctypes.data, len(m)))

    def process_node(self, seq: int, odom7, lidar) -> bool:
        o = np.ascontiguousarray(odom7, dtype=np.float64)
        l = _cloud(lidar)
        done = c_int(0)
        self._ck(self.L.erasor_updater_process_node(self.h, seq, o.ctypes.data_as(POINTER(c_double)), l.ctypes.data, len(l), PTR_HOST, ctypes.byref(done)))
        return bool(done.value)

    def prefetch_scan_ptr(self, lidar_ptr: int, n: int, ptr_kind: int):
        """Look-ahead: start the upload + voxelisation of the NEXT processed node's scan (consumed by the process_node_ptr call
        that is given the same pointer and size)."""
        self._ck(self.L.erasor_updater_prefetch_scan(self.h, c_void_p(lidar_ptr), n, ptr_kind))

    def process_node_ptr(self, seq: int, odom7, lidar_ptr: int, n: int, ptr_kind: int) -> bool:
        o = np.ascontiguousarray(odom7, dtype=np.float64)
        done = c_int(0)
        self._ck(self.L.erasor_updater_process_node(self.h, seq, o.ctypes.data_as(POINTER(c_double)), c_void_p(lidar_ptr), n, ptr_kind, ctypes.byref(done)))
        return bool(done.value)

    def cloud(self, which: int) -> np.ndarray:
        n = c_size_t(0)
        self._ck(self.L.erasor_updater_get_cloud(self.h, which, None, 0, ctypes.byref(n), PTR_HOST))
        out = np.empty((n.value, 4), dtype=np.float32)
        if n.value:
            self._ck(self.L.erasor_updater_get_cloud(self.h, which, out.ctypes.data, n.value, ctypes.byref(n), PTR_HOST))
        return out

    def map_size(self) -> int:
        n = c_size_t(0)
        self._ck(self.L.erasor_updater_map_size(self.h, ctypes.byref(n)))
        return n.value

    def save_static_map(self, voxel_size: float) -> np.ndarray:
        n = c_size_t(0)
        self._ck(self.L.erasor_updater_save_static_map(self.h, voxel_size, None, 0, ctypes.byref(n)))
        out = np.empty((n.value, 4), dtype=np.float32)
        if n.value:
            self._ck(self.L.erasor_updater_save_static_map(self.h, voxel_size, out.ctypes.data, n.value, ctypes.byref(n)))
        return out

    def voxelize(self, cloud, leaf: float) -> np.ndarray:
        c = _cloud(cloud)
        out = np.empty((max(len(c), 1), 4), dtype=np.float32)
        n = c_size_t(0)
        self._ck(self.L.erasor_updater_voxelize(self.h, c.ctypes.data, len(c), leaf, out.ctypes.data, len(out), ctypes.byref(n)))
        return out[:n.value].copy()

    def mapgen_node(self, odom7, lidar) -> np.ndarray:
        """mapgen's accumPointCloud up to cloud_curr, on the device (body cut, lift, pose, 0.2 m voxelisation)."""
        o = np.ascontiguousarray(odom7, dtype=np.float64)
        c = _cloud(lidar)
        out = np.empty((max(len(c), 1), 4), dtype=np.float32)
        n = c_size_t(0)
        self._ck(self.L.erasor_updater_mapgen_node(self.h, o.ctypes.data_as(POINTER(c_double)), c.ctypes.data, len(c), PTR_HOST, out.ctypes.data, len(out),
                                                   ctypes.byref(n)))
        return out[:n.value].copy()

    def kernel_launch_count(self) -> int:
        return int(self.L.erasor_updater_kernel_launch_count(self.h))

    def fused_profile(self):
        """Phase boundaries (ns) of the last fused prologue launch, relative to its start (include/erasor_b200.h)."""
        t = np.zeros(16, dtype=np.uint64)
        self._ck(self.L.erasor_updater_get_fused_profile(self.h, t.ctypes.data))
        return [int(x) - int(t[0]) if x else None for x in t]
