"""ctypes harness over the C ABI (include/b200slam.h) — K1, the Karto correlative scan matcher.

Mirrors the reference's ScanMatcher call sequence (Mapper.cpp:126-523) for batches:
    m = ScanMatcher(params, laser, max_batch);  m.set_scans(ranges, poses);  m.add_scans(base_ranges, base_poses)
    results = m.correlate_scan(centers, search)   |   results = m.match_scan()
There is no CPU path here: if libb200slam.so or a CUDA device is missing every call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200slam.so")
_lib = None


class B2SError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"b200slam: {abi.STATUS_NAMES.get(status, status)}: {msg}")
        self.status = status


def lib():
    """Load the product library.  Fails loudly when it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first")
    L = C.CDLL(LIB_PATH)
    dp, ip, u8p = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
    vp = C.c_void_p
    L.b2s_last_error.restype = C.c_char_p
    L.b2s_matcher_create.argtypes = [C.POINTER(abi.MatcherParams), C.POINTER(abi.Laser), C.c_int, C.c_int, C.c_int, vp,
                                     C.POINTER(vp)]
    L.b2s_matcher_destroy.argtypes = [vp]
    L.b2s_matcher_destroy.restype = None
    L.b2s_matcher_grid_info.argtypes = [vp, C.POINTER(abi.GridInfo)]
    L.b2s_matcher_set_scans.argtypes = [vp, C.c_int, dp, dp]
    L.b2s_matcher_add_scans.argtypes = [vp, C.c_int, dp, dp]
    L.b2s_matcher_set_grids.argtypes = [vp, u8p, dp]
    L.b2s_matcher_correlate_scan.argtypes = [vp, dp, C.POINTER(abi.Search), C.POINTER(abi.MatchResult)]
    L.b2s_matcher_correlate_scan_begin.argtypes = [vp, dp, C.POINTER(abi.Search), C.POINTER(abi.MatchResult)]
    L.b2s_matcher_correlate_scan_end.argtypes = [vp, C.POINTER(abi.MatchResult)]
    i32p = C.POINTER(C.c_int32)
    L.b2s_matcher_correlate_split_begin.argtypes = [vp, dp, C.POINTER(abi.Search), C.c_int, C.c_int, dp, dp, i32p]
    L.b2s_matcher_correlate_split_ties.argtypes = [vp, dp, dp]
    L.b2s_matcher_correlate_split_finish.argtypes = [vp, dp, dp, dp, C.POINTER(abi.MatchResult)]
    L.b2s_matcher_match_scan.argtypes = [vp, C.c_int, C.c_int, C.POINTER(abi.MatchResult)]
    L.b2s_matcher_match_scan_host.argtypes = [vp, C.c_int, dp, dp, C.c_int, dp, dp, C.c_int, C.c_int,
                                              C.POINTER(abi.MatchResult)]
    L.b2s_matcher_get_grid.argtypes = [vp, C.c_int, u8p, dp]
    L.b2s_matcher_get_point_readings.argtypes = [vp, C.c_int, dp]
    L.b2s_matcher_compute_offsets.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_double, ip, ip]
    L.b2s_matcher_get_response_sums.argtypes = [vp, C.c_int, ip, ip]
    L.b2s_matcher_last_timing.argtypes = [vp, dp]
    L.b2s_matcher_last_stats.argtypes = [vp, dp]
    L.b2s_matcher_last_prune_stats.argtypes = [vp, dp]
    L.b2s_matcher_sync.argtypes = [vp]
    L.b2s_matcher_set_kernel.argtypes = [vp, C.c_int]
    _lib = L
    return L


def check(status):
    if status != abi.B2S_OK:
        raise B2SError(status, lib().b2s_last_error().decode(errors="replace"))


def device_count() -> int:
    return lib().b2s_device_count()


def _d(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def results_to_arrays(res, batch):
    """-> (response[B], pose[B,3], cov[B,3,3], status[B], tie_count[B])"""
    raw = np.frombuffer(res, dtype=np.dtype([("response", "<f8"), ("pose", "<f8", 3), ("cov", "<f8", 9),
                                             ("status", "<i4"), ("tie_count", "<i4")]), count=batch)
    return (raw["response"].copy(), raw["pose"].copy(), raw["cov"].reshape(batch, 3, 3).copy(), raw["status"].copy(),
            raw["tie_count"].copy())


class ScanMatcher:
    """Batched stand-in for karto::ScanMatcher (Mapper.h:1139-1279)."""

    def __init__(self, params: abi.MatcherParams, laser: abi.Laser, max_batch: int = 1, max_base_scans: int = 1,
                 device: int = 0, stream: int | None = None):
        self.L = lib()
        self.params, self.laser = params, laser
        self.h = C.c_void_p()
        check(self.L.b2s_matcher_create(C.byref(params), C.byref(laser), device, max_batch, max_base_scans,
                                        C.c_void_p(stream) if stream else None, C.byref(self.h)))
        self.g = abi.GridInfo()
        check(self.L.b2s_matcher_grid_info(self.h, C.byref(self.g)))
        self.n = laser.n_readings
        self.batch = 0
        self.max_batch = max_batch

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.b2s_matcher_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_kernel(self, which: int):
        check(self.L.b2s_matcher_set_kernel(self.h, which))

    def set_scans(self, ranges, poses):
        r, p = f64(ranges).reshape(-1, max(self.n, 1) if self.n else 0), f64(poses).reshape(-1, 3)
        self.batch = len(p)
        self._keep = (r, p)
        check(self.L.b2s_matcher_set_scans(self.h, self.batch, _d(r), _d(p)))

    def add_scans(self, base_ranges, base_poses):
        bp = f64(base_poses).reshape(self.batch, -1, 3)
        n_base = bp.shape[1]
        br = f64(base_ranges).reshape(self.batch, n_base, self.n)
        check(self.L.b2s_matcher_add_scans(self.h, n_base, _d(br), _d(bp)))

    def pool_append(self, ranges) -> int:
        """Upload one scan's readings into the handle's device-resident scan pool; returns its row."""
        r, row = f64(ranges).reshape(self.n), C.c_int32(-1)
        self.L.b2s_matcher_pool_append.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)]
        check(self.L.b2s_matcher_pool_append(self.h, _d(r), C.byref(row)))
        return row.value

    def add_scans_pool(self, pool_rows, base_poses):
        bp = f64(base_poses).reshape(self.batch, -1, 3)
        rows = np.ascontiguousarray(pool_rows, np.int32).reshape(self.batch, bp.shape[1])
        self.L.b2s_matcher_add_scans_pool.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_double)]
        check(self.L.b2s_matcher_add_scans_pool(self.h, bp.shape[1], rows.ctypes.data_as(C.POINTER(C.c_int32)), _d(bp)))

    def set_grids(self, grids, offsets):
        g = np.ascontiguousarray(grids, dtype=np.uint8).reshape(self.batch, self.g.data_size)
        o = f64(offsets).reshape(self.batch, 2)
        check(self.L.b2s_matcher_set_grids(self.h, g.ctypes.data_as(C.POINTER(C.c_uint8)), _d(o)))

    def correlate_scan(self, centers, search: abi.Search, cov_in=None):
        c = f64(centers).reshape(self.batch, 3)
        res = (abi.MatchResult * self.batch)()
        if cov_in is not None:
            ci = f64(cov_in).reshape(self.batch, 9)
            for b in range(self.batch):
                for i in range(9):
                    res[b].cov[i] = ci[b, i]
        check(self.L.b2s_matcher_correlate_scan(self.h, _d(c), C.byref(search), res))
        return results_to_arrays(res, self.batch)

    def correlate_scan_begin(self, centers, search: abi.Search):
        """Enqueue a coarse CorrelateScan and return; pair with correlate_scan_end (two handles pipeline batches)."""
        self._pending_centers = f64(centers).reshape(self.batch, 3)  # keep the host buffer alive until _end
        check(self.L.b2s_matcher_correlate_scan_begin(self.h, _d(self._pending_centers), C.byref(search), None))

    def correlate_scan_end(self):
        res = (abi.MatchResult * self.batch)()
        check(self.L.b2s_matcher_correlate_scan_end(self.h, res))
        return results_to_arrays(res, self.batch)

    # ---- a coarse sweep whose ANGLES are split over ranks (three phases, see include/b200slam.h) ----
    def probs_len(self) -> int:
        return ((self.g.search_side + 7) & ~7) * self.g.search_side

    def split_begin(self, centers, search: abi.Search, k_first: int, k_count: int):
        """-> (best[B], probs[B, probs_len], status[B]) of angle indices [k_first, k_first + k_count)"""
        c = f64(centers).reshape(self.batch, 3)
        best = np.empty(self.batch)
        probs = np.empty((self.batch, self.probs_len()))
        status = np.empty(self.batch, dtype=np.int32)
        check(self.L.b2s_matcher_correlate_split_begin(self.h, _d(c), C.byref(search), k_first, k_count, _d(best),
                                                       _d(probs), status.ctypes.data_as(C.POINTER(C.c_int32))))
        return best, probs, status

    def split_ties(self, global_best):
        gb = f64(global_best).reshape(self.batch)
        ties = np.empty((self.batch, 5))
        check(self.L.b2s_matcher_correlate_split_ties(self.h, _d(gb), _d(ties)))
        return ties

    def split_finish(self, global_best, tie_sums, probs):
        gb, ts = f64(global_best).reshape(self.batch), f64(tie_sums).reshape(self.batch, 5)
        pr = f64(probs).reshape(self.batch, self.probs_len())
        res = (abi.MatchResult * self.batch)()
        check(self.L.b2s_matcher_correlate_split_finish(self.h, _d(gb), _d(ts), _d(pr), res))
        return results_to_arrays(res, self.batch)

    def match_scan(self, do_penalize=True, do_refine=True):
        res = (abi.MatchResult * self.batch)()
        check(self.L.b2s_matcher_match_scan(self.h, int(do_penalize), int(do_refine), res))
        return results_to_arrays(res, self.batch)

    def match_scan_host(self, ranges, poses, base_ranges, base_poses, do_penalize=True, do_refine=True):
        p = f64(poses).reshape(-1, 3)
        B = len(p)
        r = f64(ranges).reshape(B, self.n)
        bp = f64(base_poses).reshape(B, -1, 3)
        br = f64(base_ranges).reshape(B, bp.shape[1], self.n)
        res = (abi.MatchResult * B)()
        check(self.L.b2s_matcher_match_scan_host(self.h, B, _d(r), _d(p), bp.shape[1], _d(br), _d(bp), int(do_penalize),
                                                 int(do_refine), res))
        self.batch = B
        return results_to_arrays(res, B)

    def grid(self, b=0):
        out = np.zeros(self.g.data_size, dtype=np.uint8)
        off = np.zeros(2)
        check(self.L.b2s_matcher_get_grid(self.h, b, out.ctypes.data_as(C.POINTER(C.c_uint8)), _d(off)))
        return out, off

    def point_readings(self, b=0):
        out = np.zeros((self.n, 2))
        check(self.L.b2s_matcher_get_point_readings(self.h, b, _d(out)))
        return out

    def compute_offsets(self, b, angle_center, angle_offset, angle_res):
        na = abi.n_steps(angle_offset, angle_res)
        out = np.zeros((na, self.n), dtype=np.int32)
        got = C.c_int32(0)
        check(self.L.b2s_matcher_compute_offsets(self.h, b, angle_center, angle_offset, angle_res,
                                                 out.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(got)))
        assert got.value == na
        return out

    def response_sums(self, b, dims):
        """int32 [nY, nX, nAngles] of the last sweep, reference loop order."""
        ny, nx, na = dims
        out = np.zeros((ny, nx, na), dtype=np.int32)
        d = (C.c_int32 * 3)()
        check(self.L.b2s_matcher_get_response_sums(self.h, b, out.ctypes.data_as(C.POINTER(C.c_int32)), d))
        assert tuple(d) == (ny, nx, na), tuple(d)
        return out

    def last_timing(self):
        out = np.zeros(4)
        check(self.L.b2s_matcher_last_timing(self.h, _d(out)))
        return dict(lut_ms=out[0], sweep_ms=out[1], reduce_ms=out[2], path=int(out[3]))

    def last_stats(self):
        out = np.zeros(4)
        check(self.L.b2s_matcher_last_stats(self.h, _d(out)))
        return dict(empty_window_frac=out[0], path=int(out[1]), candidates=int(out[2]), beams=int(out[3]))

    def last_prune_stats(self):
        """Angle pruning of the last correlate_scan: fraction and number of (match, angle) pairs swept."""
        out = np.zeros(2)
        check(self.L.b2s_matcher_last_prune_stats(self.h, _d(out)))
        return dict(kept_frac=out[0], swept=int(out[1]))

    def sync(self):
        check(self.L.b2s_matcher_sync(self.h))
