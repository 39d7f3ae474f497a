"""ctypes harness over the C ABI — K2a (Hector log-odds map update) and K3 (Hector Gauss-Newton scan matching)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from .matcher import check, lib

_bound = False


def _bind():
    global _bound
    L = lib()
    if _bound:
        return L
    vp, fp = C.c_void_p, C.POINTER(C.c_float)
    L.b2s_hector_map_create.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, vp, C.POINTER(vp)]
    L.b2s_hector_map_destroy.argtypes = [vp]
    L.b2s_hector_map_destroy.restype = None
    L.b2s_hector_map_set_factors.argtypes = [vp, C.c_float, C.c_float]
    L.b2s_hector_map_update_by_scan.argtypes = [vp, fp, C.c_int, fp, fp]
    L.b2s_hector_map_update_by_scan_just_once.argtypes = [vp, fp, C.c_int, fp]
    L.b2s_hector_map_match_data.argtypes = [vp, fp, C.c_int, fp, C.c_int, fp, fp]
    L.b2s_hector_map_copy.argtypes = [vp, fp, C.POINTER(C.c_int32)]
    L.b2s_hector_map_copy_ros.argtypes = [vp, C.POINTER(C.c_int8)]
    L.b2s_hector_map_last_timing.argtypes = [vp, C.POINTER(C.c_double)]
    L.b2s_hector_slam_create.argtypes = [C.c_float, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, vp, C.POINTER(vp)]
    L.b2s_hector_slam_destroy.argtypes = [vp]
    L.b2s_hector_slam_destroy.restype = None
    L.b2s_hector_slam_set_update_factors.argtypes = [vp, C.c_float, C.c_float]
    L.b2s_hector_slam_set_map_update_min_diff.argtypes = [vp, C.c_float, C.c_float]
    L.b2s_hector_slam_reset.argtypes = [vp]
    L.b2s_hector_slam_update.argtypes = [vp, fp, C.c_int, fp, fp, C.c_int, fp, fp, C.POINTER(C.c_int)]
    L.b2s_hector_slam_level_dims.argtypes = [vp, C.c_int, C.POINTER(C.c_int), fp]
    L.b2s_hector_slam_copy_level.argtypes = [vp, C.c_int, fp, C.POINTER(C.c_int32)]
    L.b2s_hector_slam_copy_level_ros.argtypes = [vp, C.c_int, C.POINTER(C.c_int8)]
    L.b2s_hector_slam_stats.argtypes = [vp, C.POINTER(C.c_double)]
    ip = C.POINTER(C.c_int32)
    L.b2s_hector_slam_create_batch.argtypes = [C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int,
                                               C.c_int, vp, C.POINTER(vp)]
    L.b2s_hector_slam_set_exact.argtypes = [vp, C.c_int]
    L.b2s_hector_slam_process_stream.argtypes = [vp, C.c_int, fp, ip, fp, fp, fp, C.c_int, fp, ip, fp]
    L.b2s_hector_slam_update_batch.argtypes = [vp, fp, ip, fp, fp, C.c_int, fp, fp, ip]
    L.b2s_hector_slam_update_batch_device.argtypes = [vp, vp, vp, C.c_int, fp, vp, C.c_int]
    L.b2s_hector_slam_sync.argtypes = [vp]
    L.b2s_hector_slam_copy_level_of.argtypes = [vp, C.c_int, C.c_int, fp, ip]
    L.b2s_hector_slam_last_poses.argtypes = [vp, C.c_int, fp, fp]
    L.b2s_hector_slam_debug_set_epoch.argtypes = [vp, C.c_uint]
    L.b2s_hector_slam_match_cluster_size.argtypes = [vp]
    _bound = True
    return L


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


class HectorMap:
    """Stand-in for hectorslam::GridMap (+ its OccGridMapUtil / ScanMatcher) on one pyramid level."""

    def __init__(self, size_x, size_y, resolution, start_x=0.5, start_y=0.5, device=0, stream=None):
        self.L = _bind()
        self.sx, self.sy, self.resolution = size_x, size_y, resolution
        self.h = C.c_void_p()
        check(self.L.b2s_hector_map_create(size_x, size_y, resolution, start_x, start_y, device,
                                           C.c_void_p(stream) if stream else None, C.byref(self.h)))

    def set_factors(self, update_free, update_occupied):
        check(self.L.b2s_hector_map_set_factors(self.h, update_free, update_occupied))

    def update_by_scan(self, points, origo, world_pose):
        p = f32(points).reshape(-1, 2)
        check(self.L.b2s_hector_map_update_by_scan(self.h, _f(p), len(p), _f(f32(origo)), _f(f32(world_pose))))

    def update_by_scan_just_once(self, points_m, origo):
        """OccGridMapBase::updateByScanJustOnce (OccGridMapBase.h:175-217): points in metres, map pose (800, 800, 0)"""
        p = f32(points_m).reshape(-1, 2)
        check(self.L.b2s_hector_map_update_by_scan_just_once(self.h, _f(p), len(p), _f(f32(origo))))

    def match_data(self, points, begin_world_pose, max_iterations):
        p = f32(points).reshape(-1, 2)
        pose, cov = np.zeros(3, np.float32), np.zeros(9, np.float32)
        check(self.L.b2s_hector_map_match_data(self.h, _f(p), len(p), _f(f32(begin_world_pose)), max_iterations,
                                               _f(pose), _f(cov)))
        return pose, cov.reshape(3, 3)

    def cells(self):
        lo = np.zeros(self.sx * self.sy, np.float32)
        ui = np.zeros(self.sx * self.sy, np.int32)
        check(self.L.b2s_hector_map_copy(self.h, _f(lo), ui.ctypes.data_as(C.POINTER(C.c_int32))))
        return lo.reshape(self.sy, self.sx), ui.reshape(self.sy, self.sx)

    def ros_map(self):
        out = np.zeros((self.sy, self.sx), np.int8)
        check(self.L.b2s_hector_map_copy_ros(self.h, out.ctypes.data_as(C.POINTER(C.c_int8))))
        return out

    def last_timing(self):
        out = np.zeros(2)
        check(self.L.b2s_hector_map_last_timing(self.h, out.ctypes.data_as(C.POINTER(C.c_double))))
        return dict(update_ms=out[0], match_ms=out[1])

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.b2s_hector_map_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HectorSlam:
    """Stand-in for hectorslam::HectorSlamProcessor (slam_main/HectorSlamProcessor.h): same constructor arguments,
    update() = multi-level matchData + gated updateByScan, one call per LaserScan."""

    def __init__(self, resolution=0.05, size_x=1024, size_y=1024, start=(0.5, 0.5), levels=3,
                 update_free=0.4, update_occupied=0.9, min_dist=0.4, min_angle=0.13, device=0, stream=None,
                 batch=None, max_points=2048, exact=True):
        self.L = _bind()
        self.levels = levels
        self.batch, self.cap = batch, max_points
        self.h = C.c_void_p()
        if batch is None:
            check(self.L.b2s_hector_slam_create(resolution, size_x, size_y, start[0], start[1], levels, device,
                                                C.c_void_p(stream) if stream else None, C.byref(self.h)))
            self.cap = 2048
        else:  # B independent processors (robots / maps) behind one handle
            check(self.L.b2s_hector_slam_create_batch(batch, max_points, resolution, size_x, size_y, start[0], start[1],
                                                      levels, device, C.c_void_p(stream) if stream else None,
                                                      C.byref(self.h)))
        check(self.L.b2s_hector_slam_set_update_factors(self.h, update_free, update_occupied))
        check(self.L.b2s_hector_slam_set_map_update_min_diff(self.h, min_dist, min_angle))
        if not exact:
            check(self.L.b2s_hector_slam_set_exact(self.h, 0))
        self.map_updated = False

    def set_exact(self, exact):
        check(self.L.b2s_hector_slam_set_exact(self.h, int(bool(exact))))

    def cluster_size(self):
        """CTAs sharing the fast mode's match (1 = no cluster launch)."""
        return int(self.L.b2s_hector_slam_match_cluster_size(self.h))

    def process_stream(self, scans, origo, first_hint=None, pose_hints=None, map_without_matching=False):
        """A whole stream of LaserScans in one call (hint of scan i = pose of scan i-1, as the node's loop chains them,
        unless pose_hints gives one per scan).  Returns poses [n,3], updated flags [n], last covariance [3,3]."""
        n = len(scans)
        cnt = np.array([len(s) for s in scans], np.int32)
        cat = f32(np.concatenate([f32(s).reshape(-1, 2) for s in scans], 0)) if n else np.zeros((0, 2), np.float32)
        poses, upd, cov = np.zeros((n, 3), np.float32), np.zeros(n, np.int32), np.zeros(9, np.float32)
        fh = f32(first_hint) if first_hint is not None else None
        ph = f32(pose_hints) if pose_hints is not None else None
        check(self.L.b2s_hector_slam_process_stream(self.h, n, _f(cat), cnt.ctypes.data_as(C.POINTER(C.c_int32)),
                                                    _f(f32(origo)), _f(fh) if fh is not None else None,
                                                    _f(ph) if ph is not None else None, int(map_without_matching),
                                                    _f(poses), upd.ctypes.data_as(C.POINTER(C.c_int32)), _f(cov)))
        return poses, upd.astype(bool), cov.reshape(3, 3)

    def update_batch(self, scans, origo, pose_hints, map_without_matching=False):
        """One scan per processor of a batched handle.  scans: list of B [n_b, 2] arrays."""
        B = self.batch
        pts = np.zeros((B, self.cap, 2), np.float32)
        cnt = np.zeros(B, np.int32)
        for b, s_ in enumerate(scans):
            s_ = f32(s_).reshape(-1, 2)
            pts[b, :len(s_)] = s_
            cnt[b] = len(s_)
        poses, covs, upd = np.zeros((B, 3), np.float32), np.zeros((B, 9), np.float32), np.zeros(B, np.int32)
        ph = f32(pose_hints) if pose_hints is not None else None
        check(self.L.b2s_hector_slam_update_batch(self.h, _f(pts), cnt.ctypes.data_as(C.POINTER(C.c_int32)), _f(f32(origo)),
                                                  _f(ph) if ph is not None else None, int(map_without_matching), _f(poses),
                                                  _f(covs), upd.ctypes.data_as(C.POINTER(C.c_int32))))
        return poses, covs.reshape(B, 3, 3), upd.astype(bool)

    def update_batch_device(self, d_points, d_counts, max_n, origo, d_hints, map_without_matching=False):
        check(self.L.b2s_hector_slam_update_batch_device(self.h, C.c_void_p(d_points), C.c_void_p(d_counts), int(max_n),
                                                         _f(f32(origo)), C.c_void_p(d_hints) if d_hints else None,
                                                         int(map_without_matching)))

    def sync(self):
        check(self.L.b2s_hector_slam_sync(self.h))

    def level_of(self, b, i):
        sx, sy, _ = self.level_dims(i)
        lo, ui = np.zeros(sx * sy, np.float32), np.zeros(sx * sy, np.int32)
        check(self.L.b2s_hector_slam_copy_level_of(self.h, b, i, _f(lo), ui.ctypes.data_as(C.POINTER(C.c_int32))))
        return lo.reshape(sy, sx), ui.reshape(sy, sx)

    def last_poses(self, b=0):
        a, u = np.zeros(3, np.float32), np.zeros(3, np.float32)
        check(self.L.b2s_hector_slam_last_poses(self.h, b, _f(a), _f(u)))
        return a, u

    def debug_set_epoch(self, updates):
        check(self.L.b2s_hector_slam_debug_set_epoch(self.h, int(updates)))

    def update(self, points, origo, pose_hint, map_without_matching=False):
        p = f32(points).reshape(-1, 2)
        pose, cov, upd = np.zeros(3, np.float32), np.zeros(9, np.float32), C.c_int(0)
        check(self.L.b2s_hector_slam_update(self.h, _f(p), len(p), _f(f32(origo)), _f(f32(pose_hint)),
                                            int(map_without_matching), _f(pose), _f(cov), C.byref(upd)))
        self.map_updated = bool(upd.value)
        return pose, cov.reshape(3, 3)

    def reset(self):
        check(self.L.b2s_hector_slam_reset(self.h))

    def level_dims(self, i):
        dims, cl = (C.c_int * 2)(), C.c_float(0)
        check(self.L.b2s_hector_slam_level_dims(self.h, i, dims, C.byref(cl)))
        return dims[0], dims[1], cl.value

    def level(self, i):
        sx, sy, _ = self.level_dims(i)
        lo, ui = np.zeros(sx * sy, np.float32), np.zeros(sx * sy, np.int32)
        check(self.L.b2s_hector_slam_copy_level(self.h, i, _f(lo), ui.ctypes.data_as(C.POINTER(C.c_int32))))
        return lo.reshape(sy, sx), ui.reshape(sy, sx)

    def ros_map(self, i=0):
        sx, sy, _ = self.level_dims(i)
        out = np.zeros((sy, sx), np.int8)
        check(self.L.b2s_hector_slam_copy_level_ros(self.h, i, out.ctypes.data_as(C.POINTER(C.c_int8))))
        return out

    def stats(self):
        out = np.zeros(5)
        check(self.L.b2s_hector_slam_stats(self.h, out.ctypes.data_as(C.POINTER(C.c_double))))
        return dict(matched=int(out[0]), updated=int(out[1]), cell_visits=int(out[2]), match_ms=out[3], update_ms=out[4])

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.b2s_hector_slam_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scan_to_data_container(ranges, laser, resolution, max_dist=20.0, min_dist=0.4):
    """HectorMappingRos::rosPointCloudToDataContainer (hector_slam.cc:320-362) for a laser mounted at the base_link
    origin: beam endpoints in the laser frame (float32), filtered by squared distance, scaled by 1/resolution."""
    i = np.arange(laser.n_readings)
    ang = (laser.min_angle + i * laser.angular_resolution).astype(np.float32)
    r = np.asarray(ranges, dtype=np.float32)
    ok = np.isfinite(r)
    x = np.where(ok, r * np.cos(ang), 0).astype(np.float32)
    y = np.where(ok, r * np.sin(ang), 0).astype(np.float32)
    d2 = x * x + y * y
    keep = ok & (d2 > np.float32(min_dist * min_dist)) & (d2 < np.float32(max_dist * max_dist))
    keep &= ~((x < 0) & (d2 < 0.5))
    scale = np.float32(1.0) / np.float32(resolution)
    return np.stack([x[keep] * scale, y[keep] * scale], axis=1).astype(np.float32)
