"""Host-side mirror of the reference's registration plug-in interface, over the C ABI.

`Registration` mirrors RegistrationInterface (include/registration/registration_interface.h:11-20 upstream):
`Match(cluster, T) -> bool` (T in-out), `AddCloudToLocalMap([cloud, ...])`, `GetFitnessScore(max_range)`.
`create_matcher(mode_string, ...)` mirrors the factory branches of FrontEnd::InitMatcher
(src/slam/frontend.cpp:30-88 upstream) keyed by the same mode strings (constant_variable.h:21-25).
Clouds are numpy float32 arrays: (n,4) packed x,y,z,intensity or (n,8) pcl::PointXYZI records.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _abi
from ._abi import FlsConfig, FlsIterLog, FlsMapInfo, FlsMatchStats
from ._lib import check, lib


@dataclass
class PointcloudCluster:
    """The members of PointcloudCluster (include/lidar/pointcloud_cluster.h:13-26 upstream) a matcher reads."""
    ordered_cloud: np.ndarray | None = None
    planar_cloud: np.ndarray | None = None
    corner_cloud: np.ndarray | None = None
    point_depth_vec: np.ndarray | None = None
    point_col_index_vec: np.ndarray | None = None
    row_start_index_vec: np.ndarray | None = None
    row_end_index_vec: np.ndarray | None = None
    timestamp: int = 0
    extra: dict = field(default_factory=dict)


def _cloud(a):
    if a is None:
        return None, 0, 16, None
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (4, 8):
        raise ValueError("cloud must be (n,4) packed xyzi or (n,8) pcl::PointXYZI records")
    return a.ctypes.data_as(C.c_void_p), a.shape[0], a.shape[1] * 4, a


def _pack(clouds):
    """Host clouds -> (pointer array, count array, stride, arrays that must stay alive while the device may read them)."""
    ptrs, ns, keep, stride = [], [], [], None
    for c in clouds:
        p, n, s, a = _cloud(c)
        if stride is not None and s != stride:
            raise ValueError("all clouds of one call must share a layout")
        stride = s
        ptrs.append(p)
        ns.append(n)
        keep.append(a)
    return (C.c_void_p * len(ptrs))(*ptrs), (C.c_size_t * len(ns))(*ns), stride, keep


def _pack_device(d_ptrs, ns):
    return (C.c_void_p * len(d_ptrs))(*[int(p) for p in d_ptrs]), (C.c_size_t * len(ns))(*[int(n) for n in ns])


def _colmajor(Ts):
    """(B,4,4) poses -> a new float64 array holding each pose in Eigen's column-major memory order."""
    return np.transpose(np.asarray(Ts, np.float64), (0, 2, 1)).copy()


def _batch_out(B):
    return (C.c_int * B)(), (FlsMatchStats * B)()


class Registration:
    def __init__(self, cfg: FlsConfig):
        self.cfg = cfg
        self._h = C.c_void_p()
        check(lib().fls_create(C.byref(cfg), C.byref(self._h)), "fls_create")
        self.last_stats = FlsMatchStats()

    # -- RegistrationInterface ----------------------------------------------------------------------------
    def AddCloudToLocalMap(self, cloud_list) -> None:
        if isinstance(cloud_list, np.ndarray):
            cloud_list = [cloud_list]
        arr_p, arr_n, stride, keep = _pack(cloud_list)
        check(lib().fls_add_cloud(self._h, len(arr_p), arr_p, arr_n, stride), "fls_add_cloud")

    def Match(self, cluster: PointcloudCluster, T: np.ndarray) -> bool:
        """T: (4,4) float64, updated in place (also on failure, as upstream)."""
        po, no, so, ko = _cloud(cluster.ordered_cloud)
        pp, npl, sp, kp = _cloud(cluster.planar_cloud)
        pc, nc, scn, kc = _cloud(cluster.corner_cloud)
        strides = {s for s, k in ((so, ko), (sp, kp), (scn, kc)) if k is not None}
        if len(strides) > 1:
            raise ValueError("all clouds of one cluster must share a layout")
        stride = strides.pop() if strides else 16
        Tc = np.ascontiguousarray(np.asarray(T, np.float64).T).copy()  # Eigen column-major memory
        conv = C.c_int(0)
        st = FlsMatchStats()
        rc = lib().fls_match(self._h, po, no, pp, npl, pc, nc, stride, Tc.ctypes.data_as(C.c_void_p), C.byref(conv), C.byref(st))
        check(rc, "fls_match")
        T[...] = Tc.T
        self.last_stats = st
        return bool(conv.value)

    def GetFitnessScore(self, max_range: float) -> float:
        out = C.c_float(0)
        rc = lib().fls_fitness(self._h, float(max_range), C.byref(out))
        if rc == _abi.FLS_ERR_UNSUPPORTED:
            return float(np.finfo(np.float32).max)
        check(rc, "fls_fitness")
        return float(out.value)

    # -- batched Match (throughput entry: LoamPointToPlaneIVOX, IncrementalNDT, IcpOptimized, LoamPointToPlaneKdtree) ------
    def match_batch(self, scans, Ts):
        """scans: list of (n,4)/(n,8) host clouds — the planar clouds for the LOAM point-to-plane plug-ins (iVox and kd-tree), the
        ordered clouds for NDT and ICP; Ts: (B,4,4) float64 initial poses.  Returns (converged[B], T[B,4,4]);
        self.last_batch_stats holds the per-scan fls_match_stats (call-level timings on element 0).  More than one scan needs
        localization mode; LoamFull has no batch entry.  GetFitnessScore afterwards scores scan 0 at its final pose."""
        arr_p, arr_n, stride, keep = _pack(scans)
        Tc, (conv, st) = _colmajor(Ts), _batch_out(len(scans))
        check(lib().fls_match_batch(self._h, len(scans), arr_p, arr_n, stride, Tc.ctypes.data_as(C.c_void_p), conv, st), "fls_match_batch")
        return self._batch_result(Tc, conv, st)

    def match_batch_begin(self, scans, Ts) -> None:
        """First half of match_batch: enqueue copies + matching + read-back on the handle's stream, do not wait (the scans should sit
        in pinned host memory).  With two handles the copy of one batch overlaps the kernels of the other."""
        arr_p, arr_n, stride, keep = _pack(scans)
        Tc = _colmajor(Ts)
        self._pending = (keep, arr_p, arr_n, Tc, len(scans))  # the asynchronous copies read these until match_batch_end
        check(lib().fls_match_batch_begin(self._h, len(scans), arr_p, arr_n, stride, Tc.ctypes.data_as(C.c_void_p)), "fls_match_batch_begin")

    def match_batch_begin_device(self, d_ptrs, ns, Ts) -> None:
        """match_batch_begin with device-resident packed float4 scans."""
        arr_p, arr_n = _pack_device(d_ptrs, ns)
        Tc = _colmajor(Ts)
        self._pending = ((), arr_p, arr_n, Tc, len(d_ptrs))
        check(lib().fls_match_batch_begin_device(self._h, len(d_ptrs), arr_p, arr_n, Tc.ctypes.data_as(C.c_void_p)), "fls_match_batch_begin_device")

    def match_batch_end(self):
        keep, arr_p, arr_n, Tc, B = self._pending
        conv, st = _batch_out(B)
        check(lib().fls_match_batch_end(self._h, Tc.ctypes.data_as(C.c_void_p), conv, st), "fls_match_batch_end")
        self._pending = None
        return self._batch_result(Tc, conv, st)

    def match_batch_device(self, d_ptrs, ns, Ts):
        """Same with device-resident packed float4 scans: d_ptrs = list of device addresses, ns = point counts.  Same plug-ins and
        clouds as match_batch."""
        arr_p, arr_n = _pack_device(d_ptrs, ns)
        Tc, (conv, st) = _colmajor(Ts), _batch_out(len(d_ptrs))
        check(lib().fls_match_batch_device(self._h, len(d_ptrs), arr_p, arr_n, Tc.ctypes.data_as(C.c_void_p), conv, st), "fls_match_batch_device")
        return self._batch_result(Tc, conv, st)

    def _batch_result(self, Tc, conv, st):
        self.last_batch_stats = list(st)
        self.last_stats = st[0]
        return np.array(conv[:], bool), np.transpose(Tc, (0, 2, 1)).copy()

    def set_result_buffer_device(self, d_ptr: int, capacity_scans: int) -> None:
        """Every later Match also writes {column-major pose, converged, iterations} (18 doubles per scan) to this device
        buffer from inside the GN kernel — the input of the per-batch pose all-gather (parallel.py)."""
        check(lib().fls_set_result_buffer_device(self._h, C.c_void_p(d_ptr) if d_ptr else None, int(capacity_scans)), "fls_set_result_buffer_device")

    # -- device-resident scan (bench `value` leg) ---------------------------------------------------------
    def match_device(self, d_ptr: int, n: int, T: np.ndarray) -> bool:
        Tc = np.ascontiguousarray(np.asarray(T, np.float64).T).copy()
        conv = C.c_int(0)
        st = FlsMatchStats()
        check(lib().fls_match_device(self._h, C.c_void_p(d_ptr), n, Tc.ctypes.data_as(C.c_void_p), C.byref(conv), C.byref(st)), "fls_match_device")
        T[...] = Tc.T
        self.last_stats = st
        return bool(conv.value)

    # -- localization-mode map path (Localization::LoadLocalMap upstream) ---------------------------------
    def set_global_map(self, cloud: np.ndarray) -> None:
        p, n, s, keep = _cloud(cloud)
        check(lib().fls_set_global_map(self._h, p, n, s), "fls_set_global_map")

    def update_local_map(self, T: np.ndarray):
        """Re-cut the +-100 m local map around T when needed and hand it to the plug-in; returns (updated, n_local_points)."""
        Tc = np.ascontiguousarray(np.asarray(T, np.float64).T).copy()
        upd, nl = C.c_int(0), C.c_size_t(0)
        check(lib().fls_update_local_map(self._h, Tc.ctypes.data_as(C.c_void_p), C.byref(upd), C.byref(nl)), "fls_update_local_map")
        return bool(upd.value), int(nl.value)

    # -- introspection ---------------------------------------------------------------------------------
    def map_points(self) -> np.ndarray:
        """(n, 4) float32 points of the LOAM-iVox map, insertion order."""
        cap = max(int(self.map_info().n_points), 1)
        out = np.zeros((cap, 4), np.float32)
        n = C.c_size_t(0)
        check(lib().fls_get_map_points(self._h, out.ctypes.data_as(C.c_void_p), cap, C.byref(n)), "fls_get_map_points")
        return out[:min(cap, n.value)]

    def voxel_keys(self) -> np.ndarray:
        """(n, 3) int32 voxel keys the map currently holds (NDT / LOAM-iVox), unordered."""
        cap = max(int(self.map_info().n_voxels), 1)
        out = np.zeros((cap, 3), np.int32)
        n = C.c_size_t(0)
        check(lib().fls_get_voxel_keys(self._h, out.ctypes.data_as(C.c_void_p), cap, C.byref(n)), "fls_get_voxel_keys")
        return out[:min(cap, n.value)]

    def iter_log(self):
        cap = max(1, self.cfg.max_iterations)
        buf = (FlsIterLog * cap)()
        n = lib().fls_get_iter_log(self._h, buf, cap)
        if n < 0:
            check(n, "fls_get_iter_log")
        return [dict(H=np.array(b.H).reshape(6, 6), g=np.array(b.g), dx=np.array(b.dx), sum_residual=b.sum_residual, n_valid=b.n_valid)
                for b in buf[:n]]

    def map_info(self) -> FlsMapInfo:
        mi = FlsMapInfo()
        check(lib().fls_get_map_info(self._h, C.byref(mi)), "fls_get_map_info")
        return mi

    def ivox_add_points(self, pts: np.ndarray) -> None:
        """IVoxMap::AddPoints: append map-frame points (LRU at ivox_capacity), no insertion rule."""
        p, n, s, keep = _cloud(pts)
        check(lib().fls_ivox_add_points(self._h, p, n, s), "fls_ivox_add_points")

    def ivox_knn(self, queries: np.ndarray, k: int = 5):
        p, n, s, keep = _cloud(queries)
        out = np.zeros((n, k, 4), np.float32)
        cnt = np.zeros(n, np.int32)
        check(lib().fls_ivox_knn(self._h, p, n, s, k, out.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p)), "fls_ivox_knn")
        return out, cnt

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().fls_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def create_matcher(mode: str, **params) -> Registration:
    """Factory keyed by the reference's mode strings ("PointToPlane_IVOX", "IncrementalNDT", "IcpOptimized", ...)."""
    if mode not in _abi.METHOD_BY_MODE_STRING:
        raise ValueError(f"unknown registration_and_searcher_mode {mode!r}")
    return Registration(_abi.default_config(_abi.METHOD_BY_MODE_STRING[mode], **params))


def voxel_grid(points: np.ndarray, leaf: float, device: int = 0) -> np.ndarray:
    """VoxelGridCloud (include/common/pointcloud_utility.h:216-224 upstream) on the device."""
    p, n, s, keep = _cloud(points)
    out = np.empty((max(n, 1), 4), np.float32)
    n_out = C.c_size_t(0)
    check(lib().fls_voxel_grid(device, p, n, s, float(leaf), out.ctypes.data_as(C.c_void_p), C.byref(n_out)), "fls_voxel_grid")
    return out[:n_out.value].copy()


def pcd_write(path: str, cloud: np.ndarray) -> None:
    """pcl::io::savePCDFileBinary of an x y z intensity cloud."""
    c = np.ascontiguousarray(cloud, np.float32)
    assert c.ndim == 2 and c.shape[1] == 4
    check(lib().fls_pcd_write(str(path).encode(), c.ctypes.data_as(C.c_void_p), len(c)), "fls_pcd_write")


def pcd_read(path: str) -> np.ndarray:
    """pcl::io::loadPCDFile into packed x y z intensity records."""
    n = C.c_size_t(0)
    check(lib().fls_pcd_read(str(path).encode(), None, 0, C.byref(n)), "fls_pcd_read")
    out = np.zeros((max(n.value, 1), 4), np.float32)
    check(lib().fls_pcd_read(str(path).encode(), out.ctypes.data_as(C.c_void_p), n.value, C.byref(n)), "fls_pcd_read")
    return out[:n.value]
