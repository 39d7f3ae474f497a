"""The C restatement against the reference build (oracle/_ref/libkarto_ref.so = the unmodified open_karto sources,
compiled by `make -C oracle ref`) on fresh seeded inputs; where that build is absent, against its recorded answers
(tests/reference_replay.py).  CPU only."""
import numpy as np
import pytest

from oracle import port, ref
from reference_replay import same

D = 0.01745329251994329577


def check_result(r, res, tol=1e-12):
    pr = port.result_tuple(res)
    assert abs(r[0] - pr[0]) <= tol
    assert np.allclose(r[1], pr[1], rtol=0, atol=tol)
    assert np.allclose(r[2], pr[2], rtol=0, atol=tol)


@pytest.mark.parametrize("seed,dropout", [(20, 0.0), (21, 0.0), (22, 0.02)])
def test_cfg1_live(pkg, reference, seed, dropout):
    abi, synth = pkg.abi, pkg.synth
    mc = synth.make_match_case(seed, dropout=dropout)
    s = reference.new(ref.RefSession, ref.default_matcher_params(1.5, 0.05, 0.03, 9.25), mc.laser)
    b, c = s.add_scan(mc.base_ranges, mc.base_pose), s.add_scan(mc.ranges, mc.odom_pose)
    s.set_grid_from_scans(c, [b])
    pm = port.PortMatcher(abi.matcher_params(1.5, 0.05, 0.03, 9.25), abi.laser_from(mc.laser))
    pm.set_scan(mc.ranges, mc.odom_pose)
    pm.add_scans(mc.base_ranges, mc.base_pose)
    assert same(pm.pts, s.point_readings(c), equal_nan=True)
    assert same(pm.grid, s.grid())
    sp = s.sensor_pose(c)
    A, R = 22.5 * D, 0.25 * D
    assert same(pm.compute_offsets(sp[2], A, R), s.compute_offsets(c, sp[2], A, R))
    for pen in (True, False):
        rc, res = pm.correlate_scan(sp, abi.Search(0.75, 0.75, 0.05, 0.05, A, R, int(pen), 0), want_sums=pen)
        assert rc == 0
        check_result(s.correlate_scan(c, sp, (0.75, 0.75), (0.05, 0.05), A, R, pen, False), res)
        if pen:
            assert same(pm.last_sums, s.response_sums(c, sp, (0.75, 0.75), (0.05, 0.05), A, R))
    rc, res = pm.match_scan(mc.ranges, mc.odom_pose, mc.base_ranges, mc.base_pose)
    check_result(s.match_scan(c, [b]), res)


@pytest.mark.parametrize("res,smear,search", [(0.025, 0.03, 0.5), (0.1, 0.3, 1.0), (0.05, 0.1, 0.4)])
def test_other_geometries_live(pkg, reference, res, smear, search):
    """cfg-4 style 0.025 m grid, the outdoor yaml's 0.1 m / smear 0.3 (13x13 kernel), and a mid case."""
    abi, synth = pkg.abi, pkg.synth
    laser = synth.Laser(range_threshold=6.0)
    mc = synth.make_match_case(31, laser, max_xy=0.1, max_th_deg=4)
    s = reference.new(ref.RefSession, ref.default_matcher_params(search, res, smear, 6.0), laser)
    b, c = s.add_scan(mc.base_ranges, mc.base_pose), s.add_scan(mc.ranges, mc.odom_pose)
    pm = port.PortMatcher(abi.matcher_params(search, res, smear, 6.0), abi.laser_from(laser))
    assert same(pm.kernel(), s.kernel())
    rc, res_p = pm.match_scan(mc.ranges, mc.odom_pose, mc.base_ranges, mc.base_pose)
    r = s.match_scan(c, [b])
    assert same(pm.grid, s.grid())
    check_result(r, res_p)
    rc, res_p = pm.match_scan(mc.ranges, mc.odom_pose, mc.base_ranges, mc.base_pose, do_penalize=False,
                              do_refine=False)
    check_result(s.match_scan(c, [b], False, False), res_p)


def test_empty_grid_all_ties_live(pkg, reference):
    """No base scans: every response is 0, every candidate ties, the mean is the search centre and the
    covariance takes the MAX_VARIANCE branch (Mapper.cpp:545-552)."""
    abi, synth = pkg.abi, pkg.synth
    laser = synth.Laser(range_threshold=6.0)
    mc = synth.make_match_case(40, laser)
    s = reference.new(ref.RefSession, ref.default_matcher_params(0.5, 0.05, 0.03, 6.0), laser)
    c = s.add_scan(mc.ranges, mc.odom_pose)
    pm = port.PortMatcher(abi.matcher_params(0.5, 0.05, 0.03, 6.0), abi.laser_from(laser))
    rc, res = pm.match_scan(mc.ranges, mc.odom_pose, np.zeros((0, 1081)), np.zeros((0, 3)))
    check_result(s.match_scan(c, []), res)
    assert res.tie_count == 3 * 3 * abi.n_steps(0.5 * 2 * D, 0.2 * D)


def test_occupancy_grid_live(pkg, reference):
    abi, synth = pkg.abi, pkg.synth
    laser = synth.Laser()
    world, poses, ranges = synth.make_trajectory(3, 10, laser, step_xy=0.3, step_th_deg=8)
    ranges[4, ::50] = np.nan
    ranges[5, ::70] = np.inf
    ranges[6, ::90] = 0.05
    s = reference.new(ref.RefSession, ref.default_matcher_params(1.5, 0.05, 0.03, 9.25), laser)
    ids = [s.add_scan(ranges[i], poses[i]) for i in range(10)]
    og = s.occupancy_grid(ids, 0.05)
    po = port.occupancy_grid(abi.laser_from(laser), ranges, poses, 0.05)
    assert (og["width"], og["height"], og["width_step"]) == (po["width"], po["height"], po["width_step"])
    assert same(po["offset"], og["offset"])
    assert same(po["passes"], og["passes"]) and same(po["hits"], og["hits"])
    assert same(po["cells"], og["cells"])


def test_trace_line_live(reference):
    rng = np.random.default_rng(7)
    segs = [tuple(int(v) for v in rng.integers(-10, 60, size=4)) for _ in range(300)]

    def cells(trace_line):
        lines = [trace_line(50, 40, *q) for q in segs]
        return np.array([len(c) for c in lines]), np.concatenate(lines)
    n_ref, cells_ref = reference.call("trace_line x300", lambda ss: cells(ref.trace_line), segs)
    n, c = cells(port.trace_line)
    assert np.array_equal(n, n_ref) and same(c, cells_ref)
