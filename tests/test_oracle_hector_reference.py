"""CPU tests pinning the Hector restatement (oracle/hector_oracle.c) to the reference: the UNMODIFIED lesson4 headers
compiled against the Eigen stand-in (oracle/ref_hector.cpp -> oracle/_ref/libhector_ref.so where it was built, its
recorded answers elsewhere: tests/reference_replay.py) and the golden vectors that build produced (tests/golden/hector.npz).  Integers (update indices, Bresenham
cells) and float32 log-odds / poses / Hessians are compared bit for bit."""
import os

import numpy as np
import pytest

from oracle import port, ref_hector as rh
from reference_replay import same_bits

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def data_container(laser, ranges, res=0.05, max_dist=20.0, min_dist=0.4):
    """hector_slam.cc:320-362 for a laser at the base_link origin (float32 throughout)."""
    i = np.arange(laser.n_readings)
    ang = (laser.min_angle + i * laser.angular_resolution).astype(np.float32)
    r = np.asarray(ranges, np.float32)
    ok = np.isfinite(r)
    x = np.where(ok, r * np.cos(ang), 0).astype(np.float32)
    y = np.where(ok, r * np.sin(ang), 0).astype(np.float32)
    d2 = x * x + y * y
    keep = ok & (d2 > np.float32(min_dist * min_dist)) & (d2 < np.float32(max_dist * max_dist))
    return np.stack([x[keep], y[keep]], 1) * (np.float32(1.0) / np.float32(res))


def same_maps(a, b):
    (la, ua), (lb, ub) = a, b
    return same_bits(ua, ub) and same_bits(la, lb)


def test_update_by_scan_bit_exact(pkg, reference):
    laser = pkg.synth.Laser()
    for seed in range(6):
        mc = pkg.synth.make_match_case(100 + seed, dropout=0.02)
        pts = data_container(laser, mc.base_ranges)
        a, b = port.PortHectorMap(1024, 1024, 0.05), reference.new(rh.RefHectorMap, 1024, 1024, 0.05)
        a.set_factors(0.4, 0.9), b.set_factors(0.4, 0.9)
        for k in range(4):  # moving pose, sub-cell origo offsets
            pose = mc.base_pose.astype(np.float32) + np.float32(0.013 * k)
            o = (0.37 * k, -0.21 * k)
            a.update_by_scan(pts, o, pose), b.update_by_scan(pts, o, pose)
        assert same_maps(a.cells(), b.cells())
        for _ in range(30):  # saturate: the `< 50` clamp (GridMapLogOdds.h:108-114)
            a.update_by_scan(pts, (0, 0), mc.base_pose), b.update_by_scan(pts, (0, 0), mc.base_pose)
        assert same_maps(a.cells(), b.cells()) and a.cells()[0].max() >= 50.0
        a.close(), b.close()


def test_update_random_clouds_and_map_edges(reference):
    """Beams that start or end outside the map are dropped whole (OccGridMapBase.h:236-247); tiny maps, both axes."""
    rng = np.random.default_rng(3)
    for sx, sy, res in ((64, 64, 0.1), (200, 120, 0.05), (33, 257, 0.2)):
        a, b = port.PortHectorMap(sx, sy, res), reference.new(rh.RefHectorMap, sx, sy, res)
        for k in range(5):
            pts = rng.uniform(-1.2 * max(sx, sy), 1.2 * max(sx, sy), (400, 2)).astype(np.float32)
            pose = np.array([rng.uniform(-1, 1) * sx * res * 0.4, rng.uniform(-1, 1) * sy * res * 0.4,
                             rng.uniform(-np.pi, np.pi)], np.float32)
            o = rng.uniform(-3, 3, 2).astype(np.float32)
            a.update_by_scan(pts, o, pose), b.update_by_scan(pts, o, pose)
        assert same_maps(a.cells(), b.cells()) and (a.cells()[1] >= 0).sum() > 100
        a.close(), b.close()


def test_update_by_scan_just_once_bit_exact(reference):
    rng = np.random.default_rng(9)
    a, b = port.PortHectorMap(1601, 1601, 0.05), reference.new(rh.RefHectorMap, 1601, 1601, 0.05)
    for _ in range(3):
        p = rng.uniform(-25, 25, (700, 2)).astype(np.float32)
        a.update_by_scan_just_once(p, (0, 0)), b.update_by_scan_just_once(p, (0, 0))
    assert same_maps(a.cells(), b.cells())


def test_match_data_bit_exact(pkg, reference):
    laser = pkg.synth.Laser()
    converged = 0
    for seed in range(25):
        mc = pkg.synth.make_match_case(200 + seed)
        pts = data_container(laser, mc.base_ranges)
        pose = mc.base_pose.astype(np.float32)
        a, b = port.PortHectorMap(1024, 1024, 0.05), reference.new(rh.RefHectorMap, 1024, 1024, 0.05)
        a.set_factors(0.4, 0.9), b.set_factors(0.4, 0.9)
        for _ in range(3):
            a.update_by_scan(pts, (0, 0), pose), b.update_by_scan(pts, (0, 0), pose)
        rng = np.random.default_rng(seed)
        start = pose + (np.array([0.08, 0.08, 0.05]) * rng.uniform(-1, 1, 3)).astype(np.float32)
        (ea, ca), (eb, cb) = a.match_data(pts, start, 5), b.match_data(pts, start, 5)
        assert np.array_equal(ea.view(np.int32), eb.view(np.int32)), (seed, ea - eb)
        assert np.array_equal(ca.view(np.int32), cb.view(np.int32))
        converged += int(np.abs(eb[:2] - pose[:2]).max() < 0.03)  # and the reference does re-align the scan
        e0a, e0b = a.match_data(pts[:0], start, 5)[0], b.match_data(pts[:0], start, 5)[0]
        assert np.array_equal(e0a, start) and np.array_equal(e0b, start)
        a.close(), b.close()
    assert converged >= 18  # single-level Gauss-Newton has a small capture basin; most perturbed starts re-align


def run_stream(proc, laser, ranges, start_pose, first_without_matching):
    est, out = start_pose.astype(np.float32), []
    for i in range(len(ranges)):
        est, cov = proc.update(data_container(laser, ranges[i]), (0, 0), est, first_without_matching and i == 0)
        out.append(np.concatenate([est, cov.ravel()]))
    return np.array(out, np.float32)


@pytest.mark.parametrize("first_without_matching", [False, True])
def test_processor_stream_bit_exact(pkg, reference, first_without_matching):
    """HectorSlamProcessor::update over a 3-level MapRepMultiMap on a 60-scan trajectory: every pose, every Hessian
    and all three final maps equal the reference's bit for bit."""
    laser = pkg.synth.Laser()
    _, poses, ranges = pkg.synth.make_trajectory(31, 60, laser, step_xy=0.12, step_th_deg=2.0)
    kw = dict(resolution=0.05, size_x=1000, size_y=1000, start=(0.5, 0.5), levels=3, min_dist=0.15, min_angle=0.06)
    a, b = port.PortHectorProcessor(**kw), reference.new(rh.RefHectorProcessor, **kw)
    ta = run_stream(a, laser, ranges, poses[0], first_without_matching)
    tb = run_stream(b, laser, ranges, poses[0], first_without_matching)
    assert np.array_equal(ta.view(np.int32), tb.view(np.int32))
    n_updates = []
    for lvl in range(3):
        assert same_maps(a.level(lvl), b.level(lvl))
        n_updates.append((a.level(lvl)[1].max() + 1) // 3)
    assert n_updates[0] >= 4 and n_updates[0] == n_updates[1] == n_updates[2]
    assert np.abs(tb[-1, :2] - poses[-1, :2]).max() < 0.05
    a.close(), b.close()


def test_processor_angle_gate_truncates(pkg, reference):
    """UtilFunctions.h:88 calls the unqualified abs() with only <cmath> included -> int abs(int): a 0.5 rad turn does
    NOT trigger a map update with angleDiffThresh 0.13, a 1.2 rad turn does.  Restatement and reference agree."""
    laser = pkg.synth.Laser()
    mc = pkg.synth.make_match_case(7)
    pts = data_container(laser, mc.base_ranges)

    def map_updates(proc, pts, turn):
        proc.update(pts, (0, 0), np.zeros(3, np.float32), True)
        proc.update(pts, (0, 0), np.array([0, 0, turn], np.float32), False)
        n = (proc.level(0)[1].max() + 1) // 3
        proc.close()
        return n
    for turn, expect in ((0.5, 1), (1.2, 2)):
        n = [map_updates(port.PortHectorProcessor(size_x=512, size_y=512), pts, turn),
             reference.call("map updates after a turn",
                            lambda p, t: map_updates(rh.RefHectorProcessor(size_x=512, size_y=512), p, t), pts, turn)]
        assert n == [expect, expect], (turn, n)


def test_hector_golden(pkg):
    """The same comparisons against vectors the reference build produced (tests/golden/make_golden.py hector):
    runs wherever the restatement compiles, e.g. on the GPU box where /root/reference does not exist."""
    g = np.load(os.path.join(G, "hector.npz"))
    kw = dict(resolution=float(g["resolution"]), size_x=int(g["size"]), size_y=int(g["size"]), start=(0.5, 0.5), levels=3,
              min_dist=float(g["min_dist"]), min_angle=float(g["min_angle"]))
    p = port.PortHectorProcessor(**kw)
    est = g["start_pose"].astype(np.float32)
    for i in range(int(g["n_scans"])):
        est, cov = p.update(g[f"pts{i}"], (0, 0), est, bool(g["without_matching"][i]))
        assert np.array_equal(np.concatenate([est, cov.ravel()]).view(np.int32), g["trace"][i].view(np.int32)), i
    for lvl in range(3):
        lo, ui = p.level(lvl)
        idx = np.flatnonzero(ui.ravel() >= 0)
        assert np.array_equal(idx, g[f"l{lvl}_idx"])
        assert np.array_equal(ui.ravel()[idx], g[f"l{lvl}_ui"])
        assert np.array_equal(lo.ravel()[idx].view(np.int32), g[f"l{lvl}_lo"].view(np.int32))
        assert (lo.ravel()[ui.ravel() < 0] == 0).all()
    m = port.PortHectorMap(int(g["jo_size"]), int(g["jo_size"]), 0.05)
    m.update_by_scan_just_once(g["jo_pts"], (0, 0))
    lo, ui = m.cells()
    idx = np.flatnonzero(ui.ravel() >= 0)
    assert np.array_equal(idx, g["jo_idx"]) and np.array_equal(ui.ravel()[idx], g["jo_ui"])
    assert np.array_equal(lo.ravel()[idx].view(np.int32), g["jo_lo"].view(np.int32))


def test_grid_probability_double_exp(pkg, reference):
    """getGridProbability (GridMapLogOdds.h:136-140): the unqualified exp() on a float is the C library's double exp,
    rounded to float (the reference build imports `exp`, not `expf`).  2^20 log-odds values incl. every multiple-sum
    the update factors can produce: restatement == reference, bit for bit; and the expf reading would NOT be."""
    import ctypes as C
    rng = np.random.default_rng(0)
    lf, lo_ = np.float32(np.log(np.float32(0.4) / np.float32(0.6))), np.float32(np.log(np.float32(0.9) / np.float32(0.1)))
    combos = (np.arange(-60, 1, dtype=np.float32)[:, None] * lf + np.arange(0, 40, dtype=np.float32)[None, :] * lo_).ravel()
    v = np.concatenate([combos, rng.uniform(-60, 60, (1 << 20) - len(combos)).astype(np.float32)]).astype(np.float32)

    def probabilities(fn, v):
        out = np.zeros_like(v)
        fn(v.ctypes.data_as(C.POINTER(C.c_float)), len(v), out.ctypes.data_as(C.POINTER(C.c_float)))
        return out
    a = probabilities(port.lib().orc_hector_grid_probabilities, v)
    b = reference.call("grid probabilities", lambda x: probabilities(rh.lib().ref_hector_grid_probabilities, x), v)
    assert same_bits(a, b)
    with np.errstate(all="ignore"):
        odds_f = np.exp(v)  # numpy float32 exp: the other reading
        alt = odds_f / (odds_f + np.float32(1.0))
    assert (alt.view(np.int32) != a.view(np.int32)).any()  # a is b, bit for bit
