"""legkilo_b200 — thin ctypes driver over liblegkilo_b200.so (the C-ABI in include/legkilo_b200.h).

The product is the CUDA library; this module only marshals numpy buffers across the C boundary
for tests and bench.py. It never computes the hot path itself and has no CPU fallback: if the
shared library is missing, or no CUDA device is present, it raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import abi

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.normpath(os.path.join(_PKG, "..", "..", "liblegkilo_b200.so"))
HEADER_PATH = os.path.normpath(os.path.join(_PKG, "..", "..", "..", "include", "legkilo_b200.h"))

_LIB = None


class LkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"legkilo_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load the CUDA library. Fails loudly when it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        vp, i32, u32, dbl = C.c_void_p, C.c_int, C.c_uint32, C.c_double
        L.lk_create.argtypes = [vp, vp, vp, vp, i32, vp]
        L.lk_destroy.argtypes = [vp]
        L.lk_last_error.restype = C.c_char_p
        L.lk_last_error.argtypes = [vp]
        L.lk_init_process_cov.argtypes = [vp, vp]
        L.lk_state_default.argtypes = [vp]
        L.lk_host_alloc.argtypes = [vp, C.c_size_t]
        L.lk_host_free.argtypes = [vp]
        L.lk_set_param.argtypes = [vp, C.c_char_p, dbl]
        L.lk_sync.argtypes = [vp]
        L.lk_map_reserve.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64]
        L.lk_map_upload.argtypes = [vp, vp, C.c_size_t]
        L.lk_map_download.argtypes = [vp, vp, C.c_size_t, vp]
        L.lk_map_build.argtypes = [vp, vp, vp, C.c_size_t, vp, vp, vp]
        L.lk_map_stats.argtypes = [vp, vp]
        L.lk_map_slide.argtypes = [vp, vp, vp, vp]
        L.lk_tum_line.argtypes = [dbl, vp, vp, C.c_char_p, C.c_size_t]
        L.lk_scan_update.argtypes = [vp, i32] + [vp] * 9 + [i32, i32, vp, vp]
        L.lk_batch_stage.argtypes = [vp, i32] + [vp] * 9
        L.lk_batch_run.argtypes = [vp, i32, i32]
        L.lk_batch_run_range.argtypes = [vp, u32, u32, i32, i32]
        L.lk_timer_start.argtypes = [vp]
        L.lk_timer_stop.argtypes = [vp] * 5
        L.lk_debug_read.argtypes = [vp, i32, vp, C.c_size_t]
        L.lk_batch_fetch.argtypes = [vp] * 6
        L.lk_batch_last_timing.argtypes = [vp] * 5
        L.lk_debug_residuals.argtypes = [vp, vp, vp, vp, u32] + [vp] * 5
        L.lk_predict.argtypes = [vp, i32, vp, vp, vp, vp, i32, i32]
        L.lk_update_by_points.argtypes = [vp, vp, vp, u32, vp, vp, vp]
        L.lk_obs_imu.argtypes = [vp, vp, vp, vp, vp, vp, u32, dbl, dbl]
        L.lk_obs_kinimu.argtypes = [vp, vp, vp, vp, vp, vp, u32, dbl, dbl]
        L.lk_process_scan.argtypes = [vp, vp, vp, vp, vp, vp, u32, vp, vp, u32, vp, vp, u32, dbl, dbl, i32, i32, vp,
                                      vp, vp]
        L.lk_decode_pointcloud2.argtypes = [vp, vp, u32, vp, C.c_float, i32, dbl, vp, vp, vp, vp, vp]
        L.lk_preprocess_scan.argtypes = [vp, vp, u32, C.c_float, vp, vp, vp, vp, vp]
        _LIB = L
    return _LIB


def tum_line(timestamp, rot, pos) -> str:
    """TrajectorySaver::write (trajectory_saver.hpp:43-50)."""
    rot = np.ascontiguousarray(rot, np.float64).reshape(9); pos = np.ascontiguousarray(pos, np.float64)
    buf = C.create_string_buffer(256)
    n = lib().lk_tum_line(float(timestamp), _p(rot), _p(pos), buf, 256)
    if n < 0:
        raise LkError(n, "lk_tum_line")
    return buf.value.decode()


def _p(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.cast(a, C.c_void_p)


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array over cudaHostAlloc'ed (pinned) memory; freed when the array is collected."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    ptr = C.c_void_p()
    rc = lib().lk_host_alloc(C.byref(ptr), max(n, 1))
    if rc:
        raise LkError(rc, "cudaHostAlloc failed")
    buf = (C.c_char * max(n, 1)).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    class _Owner:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            try:
                lib().lk_host_free(self.p)
            except Exception:
                pass
    _OWNERS[arr.ctypes.data] = _Owner(ptr)
    return arr


_OWNERS: dict = {}


class Engine:
    """One device context: extrinsics + ESKF / map configuration + the map in HBM.
    Mirrors what KILO owns (legkilo/src/core/slam/KILO.h:48-63)."""

    def __init__(self, cfg: dict, device: int = 0):
        self.cfg = cfg
        self._ec = abi.eskf_cfg(cfg)
        self._mc = abi.map_cfg(cfg)
        R, t = abi.extrinsics(cfg)
        self._R, self._t = R, t
        self.h = C.c_void_p()
        rc = lib().lk_create(C.byref(self._ec), C.byref(self._mc), _p(R), _p(t), device, C.byref(self.h))
        if rc:
            raise LkError(rc, lib().lk_last_error(None).decode())

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            lib().lk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc:
            raise LkError(rc, lib().lk_last_error(self.h).decode())

    def set_param(self, name: str, value: float):
        self._chk(lib().lk_set_param(self.h, name.encode(), float(value)))

    # ---- map ---------------------------------------------------------------------------------
    def map_reserve(self, max_roots: int, max_nodes: int, max_points: int):
        self._chk(lib().lk_map_reserve(self.h, max_roots, max_nodes, max_points))

    def map_upload(self, blob: np.ndarray):
        blob = np.ascontiguousarray(blob, np.uint8)
        self._chk(lib().lk_map_upload(self.h, _p(blob), blob.size))

    def map_download(self) -> np.ndarray:
        sz = C.c_size_t(0)
        self._chk(lib().lk_map_download(self.h, None, 0, C.byref(sz)))
        buf = np.zeros(sz.value, np.uint8)
        self._chk(lib().lk_map_download(self.h, _p(buf), buf.size, C.byref(sz)))
        return buf[:sz.value]

    def map_build(self, xyz_world, xyz_body, R=None, rot_cov=None, pos_cov=None):
        xyz_world = np.ascontiguousarray(xyz_world, np.float32)
        xyz_body = np.ascontiguousarray(xyz_body, np.float32)
        R = np.eye(3) if R is None else np.ascontiguousarray(R, np.float64)
        rot_cov = 1e-6 * np.eye(3) if rot_cov is None else np.ascontiguousarray(rot_cov, np.float64)
        pos_cov = 1e-6 * np.eye(3) if pos_cov is None else np.ascontiguousarray(pos_cov, np.float64)
        self._chk(lib().lk_map_build(self.h, _p(xyz_world), _p(xyz_body), len(xyz_world), _p(R), _p(rot_cov),
                                     _p(pos_cov)))

    def map_slide(self, position):
        """VoxelMapManager::mapSliding (voxel_map.cc:552-571). Returns (slid, removed root voxels)."""
        pos = np.ascontiguousarray(position, np.float64)
        slid = C.c_int32(0); removed = C.c_uint64(0)
        self._chk(lib().lk_map_slide(self.h, _p(pos), C.byref(slid), C.byref(removed)))
        return bool(slid.value), int(removed.value)

    def map_stats(self):
        out = np.zeros(4, np.uint64)
        self._chk(lib().lk_map_stats(self.h, _p(out)))
        return dict(roots=int(out[0]), nodes=int(out[1]), points=int(out[2]), planes=int(out[3]))

    # ---- hot path ------------------------------------------------------------------------------
    @staticmethod
    def _norm_batch(x, P, clk, pts, scan_offsets, scan_bucket_ptr, bucket_offsets, bucket_times):
        x = np.ascontiguousarray(x, abi.STATE_DTYPE)
        batch = len(x)
        P = np.ascontiguousarray(P, np.float64).reshape(batch, 900)
        clk = np.ascontiguousarray(clk, abi.CLOCK_DTYPE)
        pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
        scan_offsets = np.ascontiguousarray(scan_offsets, np.uint32)
        if scan_bucket_ptr is None:  # one bucket per scan
            scan_bucket_ptr = np.arange(batch + 1, dtype=np.uint32)
            bucket_offsets = scan_offsets
        scan_bucket_ptr = np.ascontiguousarray(scan_bucket_ptr, np.uint32)
        bucket_offsets = np.ascontiguousarray(bucket_offsets, np.uint32)
        bucket_times = np.ascontiguousarray(bucket_times, np.float64)
        assert len(scan_offsets) == batch + 1 and len(scan_bucket_ptr) == batch + 1
        assert len(bucket_offsets) == scan_bucket_ptr[-1] + 1 and len(bucket_times) == scan_bucket_ptr[-1]
        return x, P, clk, pts, scan_offsets, scan_bucket_ptr, bucket_offsets, bucket_times

    def scan_update(self, x, P, Q, clk, pts, scan_offsets, bucket_times, scan_bucket_ptr=None, bucket_offsets=None,
                    iters=1, update_map=False, want_world=True, pinned=False):
        """lk_scan_update: host buffers in, host buffers out (copies of x / P / clk are returned).
        pinned=True puts the points and the world cloud in page-locked memory (lk_host_alloc), which lets a
        one-scan call run in direct mode (the kernel reads / writes them in place)."""
        x, P, clk, pts, so, sbp, bo, bt = self._norm_batch(x, P, clk, pts, scan_offsets, scan_bucket_ptr,
                                                           bucket_offsets, bucket_times)
        x = x.copy(); P = P.copy(); clk = clk.copy()
        Q = np.ascontiguousarray(Q, np.float64)
        if pinned:
            hp = pinned_empty(pts.shape, np.float32); hp[...] = pts; pts = hp
            world = pinned_empty((len(pts), 4), np.float32) if want_world else None
            if world is not None:
                world[...] = 0
        else:
            world = np.zeros((len(pts), 4), np.float32) if want_world else None
        neff = np.zeros(len(x), np.uint32)
        self._chk(lib().lk_scan_update(self.h, len(x), _p(x), _p(P), _p(Q), _p(clk), _p(pts), _p(so), _p(sbp), _p(bo),
                                       _p(bt), iters, int(update_map), _p(world), _p(neff)))
        return dict(x=x, P=P, clk=clk, world=world, n_eff=neff)

    def stage(self, x, P, Q, clk, pts, scan_offsets, bucket_times, scan_bucket_ptr=None, bucket_offsets=None):
        x, P, clk, pts, so, sbp, bo, bt = self._norm_batch(x, P, clk, pts, scan_offsets, scan_bucket_ptr,
                                                           bucket_offsets, bucket_times)
        Q = np.ascontiguousarray(Q, np.float64)
        self._staged = (len(x), len(pts))
        self._chk(lib().lk_batch_stage(self.h, len(x), _p(x), _p(P), _p(Q), _p(clk), _p(pts), _p(so), _p(sbp), _p(bo),
                                       _p(bt)))

    def run(self, iters=1, update_map=False):
        self._chk(lib().lk_batch_run(self.h, iters, int(update_map)))

    def run_range(self, first, count, iters=1, update_map=False):
        """Asynchronous: enqueue scans [first, first+count) of the staged batch (no host sync)."""
        self._chk(lib().lk_batch_run_range(self.h, first, count, iters, int(update_map)))

    def timer_start(self):
        self._chk(lib().lk_timer_start(self.h))

    def timer_stop(self):
        t = C.c_float(); r = C.c_float(); n = C.c_uint32(); nr = C.c_uint32()
        self._chk(lib().lk_timer_stop(self.h, C.byref(t), C.byref(r), C.byref(n), C.byref(nr)))
        return dict(total_ms=t.value, residual_ms=r.value, launches=n.value, residual_launches=nr.value)

    def sync(self):
        self._chk(lib().lk_sync(self.h))

    def fetch(self, want_world=True):
        batch, npts = self._staged
        x = np.zeros(batch, abi.STATE_DTYPE); P = np.zeros((batch, 900)); clk = np.zeros(batch, abi.CLOCK_DTYPE)
        world = np.zeros((npts, 4), np.float32) if want_world else None
        neff = np.zeros(batch, np.uint32)
        self._chk(lib().lk_batch_fetch(self.h, _p(x), _p(P), _p(clk), _p(world), _p(neff)))
        return dict(x=x, P=P, clk=clk, world=world, n_eff=neff)

    def last_timing(self):
        t = C.c_float(); r = C.c_float(); n = C.c_uint32(); nr = C.c_uint32()
        self._chk(lib().lk_batch_last_timing(self.h, C.byref(t), C.byref(r), C.byref(n), C.byref(nr)))
        return dict(total_ms=t.value, residual_ms=r.value, launches=n.value, residual_launches=nr.value)

    def debug_residuals(self, x, P, pts):
        x = np.ascontiguousarray(x, abi.STATE_DTYPE); P = np.ascontiguousarray(P, np.float64)
        pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
        n = len(pts)
        ok = np.zeros(n, np.uint8); h = np.zeros((n, 6)); z = np.zeros(n); R = np.zeros(n)
        key = np.zeros((n, 3), np.int32)
        self._chk(lib().lk_debug_residuals(self.h, _p(x), _p(P), _p(pts), n, _p(ok), _p(h), _p(z), _p(R), _p(key)))
        return dict(ok=ok, h=h, z=z, R=R, key=key)

    def debug_partials(self, n_chunks: int) -> np.ndarray:
        """Per-chunk partial rows of the last multi-kernel residual pass (lk_debug_read, what = 0): [n_chunks, 32]
        doubles, A = sum h^T h / R upper triangle row-major (21) | b = sum h z / R (6) | sum R | count | pad. The
        persistent per-scan kernel (fused, batch of one) keeps its partials elsewhere and leaves these alone."""
        out = np.zeros((n_chunks, 32))
        self._chk(lib().lk_debug_read(self.h, 0, _p(out), out.nbytes))
        return out

    def update_by_points(self, x, P, h, z, R):
        """ESKF::updateByPoints (eskf.cc:91-113) from explicit rows."""
        x = np.array(x, abi.STATE_DTYPE, copy=True); P = np.array(P, np.float64, copy=True).reshape(900)
        h = np.ascontiguousarray(h, np.float64).reshape(-1, 6); z = np.ascontiguousarray(z, np.float64)
        R = np.ascontiguousarray(R, np.float64)
        self._chk(lib().lk_update_by_points(self.h, _p(x), _p(P), len(z), _p(h), _p(z), _p(R)))
        return x, P

    def obs_imu(self, x, P, Q, clk, imu, gravity=9.81, acc_norm=1.0):
        """KILO::predictUpdateImu per sample (KILO.cc:235-258)."""
        x = np.array(x, abi.STATE_DTYPE, copy=True); P = np.array(P, np.float64, copy=True).reshape(900)
        clk = np.array(clk, abi.CLOCK_DTYPE, copy=True); Q = np.ascontiguousarray(Q, np.float64)
        imu = np.ascontiguousarray(imu, abi.IMU_DTYPE)
        self._chk(lib().lk_obs_imu(self.h, _p(x), _p(P), _p(Q), _p(clk), _p(imu), len(imu), gravity, acc_norm))
        return x, P, clk

    def obs_kinimu(self, x, P, Q, clk, kin, gravity=9.81, acc_norm=1.0):
        """KILO::predictUpdateKinImu per sample (KILO.cc:260-314)."""
        x = np.array(x, abi.STATE_DTYPE, copy=True); P = np.array(P, np.float64, copy=True).reshape(900)
        clk = np.array(clk, abi.CLOCK_DTYPE, copy=True); Q = np.ascontiguousarray(Q, np.float64)
        kin = np.ascontiguousarray(kin, abi.KINIMU_DTYPE)
        self._chk(lib().lk_obs_kinimu(self.h, _p(x), _p(P), _p(Q), _p(clk), _p(kin), len(kin), gravity, acc_norm))
        return x, P, clk

    def process_scan(self, x, P, Q, clk, pts, bucket_offsets, bucket_times, imu=None, kin=None, gravity=9.81, acc_norm=1.0,
                     iters=1, update_map=True):
        """The second lambda of KILO::process (KILO.cc:367-396) for one scan, inertial / kinematic queue
        interleaved on the device."""
        x = np.array(x, abi.STATE_DTYPE, copy=True); P = np.array(P, np.float64, copy=True).reshape(900)
        clk = np.array(clk, abi.CLOCK_DTYPE, copy=True); Q = np.ascontiguousarray(Q, np.float64)
        pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
        bo = np.ascontiguousarray(bucket_offsets, np.uint32); bt = np.ascontiguousarray(bucket_times, np.float64)
        imu = None if imu is None else np.ascontiguousarray(imu, abi.IMU_DTYPE)
        kin = None if kin is None else np.ascontiguousarray(kin, abi.KINIMU_DTYPE)
        nm = len(imu) if imu is not None else (len(kin) if kin is not None else 0)
        world = np.zeros((len(pts), 4), np.float32); neff = np.zeros(1, np.uint32); ncons = np.zeros(1, np.uint32)
        self._chk(lib().lk_process_scan(self.h, _p(x), _p(P), _p(Q), _p(clk), _p(pts), len(pts), _p(bo), _p(bt), len(bt), _p(imu),
                                        _p(kin), nm, gravity, acc_norm, iters, int(update_map), _p(world), _p(neff), _p(ncons)))
        return dict(x=x, P=P, clk=clk, world=world, n_eff=int(neff[0]), n_consumed=int(ncons[0]))

    def decode_pointcloud2(self, data, layout, blind, filter_num, time_scale):
        """lk_decode_pointcloud2: raw PointCloud2 bytes -> float4 (x, y, z, curvature) + intensity."""
        data = np.ascontiguousarray(data, np.uint8)
        n = data.size // layout.point_step
        pts = np.zeros((n, 4), np.float32); inten = np.zeros(n, np.float32)
        no = np.zeros(1, np.uint32); ft = np.zeros(1); lt = np.zeros(1)
        self._chk(lib().lk_decode_pointcloud2(self.h, _p(data), n, C.byref(layout), blind, filter_num, time_scale, _p(pts),
                                              _p(inten), _p(no), _p(ft), _p(lt)))
        return pts[:no[0]].copy(), inten[:no[0]].copy(), float(ft[0]), float(lt[0])

    def preprocess_scan(self, pts, leaf):
        """lk_preprocess_scan: voxel-grid centroid filter, stable curvature sort, bucket boundaries."""
        pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
        n = len(pts)
        out = np.zeros((n, 4), np.float32); offs = np.zeros(n + 1, np.uint32); curv = np.zeros(max(n, 1), np.float32)
        no = np.zeros(1, np.uint32); nb = np.zeros(1, np.uint32)
        self._chk(lib().lk_preprocess_scan(self.h, _p(pts), n, leaf, _p(out), _p(no), _p(offs), _p(curv), _p(nb)))
        return out[:no[0]].copy(), offs[:nb[0] + 1].copy(), curv[:nb[0]].copy()

    def predict(self, x, P, Q, dt, prop_state=True, prop_cov=True):
        x = np.array(x, abi.STATE_DTYPE, copy=True); batch = len(x)
        P = np.array(P, np.float64, copy=True).reshape(batch, 900)
        Q = np.ascontiguousarray(Q, np.float64); dt = np.ascontiguousarray(dt, np.float64)
        self._chk(lib().lk_predict(self.h, batch, _p(x), _p(P), _p(Q), _p(dt), int(prop_state), int(prop_cov)))
        return x, P
