"""CPU tests of the GMapping restatement (pinned to the reference's real headers + golden vectors) and of the
Hector restatement (semantic self-checks here; bit-exact pinning to the reference headers is in
test_oracle_hector_reference.py)."""
import os

import numpy as np

from oracle import port, ref_gmapping as rg
from reference_replay import same

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_gmapping_golden():
    g = np.load(os.path.join(G, "gmapping.npz"))
    for k in range(2):
        b = g[f"c{k}_bounds"]
        m = port.PortGMap(*b)
        assert [m.size_x, m.size_y] == list(g[f"c{k}_size"])
        assert m.compute_map(g[f"c{k}_ranges"], g["angles"], tuple(g[f"c{k}_laser_xy"])) == 0
        n, v, ax, ay = m.cells()
        ys, xs = np.nonzero(v)
        assert np.array_equal(np.stack([ys, xs], 1), g[f"c{k}_cells_yx"])
        assert np.array_equal(n[ys, xs], g[f"c{k}_n"]) and np.array_equal(v[ys, xs], g[f"c{k}_visits"])
        assert np.array_equal(ax[ys, xs], g[f"c{k}_acc_x"]) and np.array_equal(ay[ys, xs], g[f"c{k}_acc_y"])


def test_gmapping_live(pkg, reference):
    """Against the reference's grid headers (oracle/_ref/libgmapping_ref.so, or its recorded answers where that build is
    absent: tests/reference_replay.py)."""
    rng = np.random.default_rng(5)
    segs = [tuple(int(v) for v in rng.integers(0, 300, 4)) for _ in range(3000)]

    def cells(grid_line):
        lines = [grid_line(*q) for q in segs]
        return np.array([len(c) for c in lines]), np.concatenate(lines)
    n_ref, cells_ref = reference.call("grid_line x3000", lambda ss: cells(rg.grid_line), segs)
    n, c = cells(port.gmap_grid_line)
    assert np.array_equal(n, n_ref) and same(c, cells_ref)
    laser = pkg.synth.Laser()
    ang = (np.float32(laser.min_angle) + np.arange(1081, dtype=np.float32) * np.float32(laser.angular_resolution)).astype(np.float64)
    a, b = reference.new(rg.RefGMap, -25, -25, 25, 25, 0.1), port.PortGMap(-25, -25, 25, 25, 0.1)
    for seed in range(4):  # several scans accumulated into one map
        r = pkg.synth.make_match_case(50 + seed).ranges.astype(np.float32).astype(np.float64)
        assert a.compute_map(r, ang, (0.2 * seed, -0.1 * seed)) == 0
        assert b.compute_map(r, ang, (0.2 * seed, -0.1 * seed)) == 0
    for x, y in zip(a.cells()[:4], b.cells()):
        assert same(y, x)
    unknown, occupied = reference.call("occupancy classes", lambda: (a.cells()[4] < 0, a.cells()[4] > 0.25))
    ros = b.ros_map()[:b.size_y, :b.size_x]  # the 500x500 published map holds the 480x480 patch-rounded storage
    assert same(ros == -1, unknown) and same(ros == 100, occupied)
    # a ray leaving the map: the reference would assert; both report an error and change nothing
    c, d = reference.new(rg.RefGMap, -5, -5, 5, 5, 0.05), port.PortGMap(-5, -5, 5, 5, 0.05)
    assert c.compute_map(np.full(1081, 20.0), ang) == -1 and d.compute_map(np.full(1081, 20.0), ang) == -1
    assert d.visits.sum() == 0
    a.close(); c.close()


def hector_points(pkg, seed, res=0.05):
    H = pkg.load("hector") if False else None  # the harness module needs libb200slam; restate the conversion here
    laser = pkg.synth.Laser()
    mc = pkg.synth.make_match_case(seed)
    i = np.arange(1081)
    ang = (laser.min_angle + i * laser.angular_resolution).astype(np.float32)
    r = mc.base_ranges.astype(np.float32)
    x, y = (r * np.cos(ang)).astype(np.float32), (r * np.sin(ang)).astype(np.float32)
    d2 = x * x + y * y
    keep = (d2 > 0.16) & (d2 < 400.0)
    return np.stack([x[keep], y[keep]], 1) * np.float32(1.0 / res), mc.base_pose.astype(np.float32)


def test_hector_update_semantics(pkg):
    """Self-consistency of the K2a restatement: once-per-scan stamps, occupied wins over free, update indices."""
    pts, pose = hector_points(pkg, 1)
    m = port.PortHectorMap(1024, 1024, 0.05)
    m.set_factors(0.4, 0.9)
    visits = m.update_by_scan(pts, (0.0, 0.0), pose)
    lo, ui = m.cells()
    lf, locc = np.float32(np.log(np.float32(0.4) / np.float32(0.6))), np.float32(np.log(np.float32(0.9) / (np.float32(1) - np.float32(0.9))))
    assert visits > 50_000
    assert set(np.unique(ui)) <= {-1, 1, 2}
    assert np.allclose(lo[ui == 1], lf) and (ui == 1).sum() > 10_000       # freed exactly once
    occ = lo[ui == 2]
    assert ((np.abs(occ - locc) < 1e-6) | (np.abs(occ - ((lf - lf) + locc)) < 1e-6)).all() and len(occ) > 300
    assert (lo[ui == -1] == 0).all()
    # 30 more identical updates: occupied cells saturate just above 50 (the clamp stops further increments)
    for _ in range(30):
        m.update_by_scan(pts, (0.0, 0.0), pose)
    lo2, ui2 = m.cells()
    assert lo2.max() < 50.0 + locc + 1e-3 and lo2.max() >= 50.0
    assert ui2.max() == 30 * 3 + 2


def test_hector_gn_recovers_pose(pkg):
    """Self-consistency of the K3 restatement: build a map from a scan at a known pose, perturb, re-align."""
    pts, pose = hector_points(pkg, 2)
    m = port.PortHectorMap(1024, 1024, 0.05)
    m.set_factors(0.4, 0.9)
    for _ in range(3):
        m.update_by_scan(pts, (0.0, 0.0), pose)
    start = pose + np.array([0.06, -0.05, 0.03], np.float32)
    est, cov = m.match_data(pts, start, 12)
    assert np.abs(est[:2] - pose[:2]).max() < 0.02 and abs(est[2] - pose[2]) < 0.01
    assert np.allclose(cov, cov.T) and cov[0, 0] > 0 and cov[1, 1] > 0
    est0, _ = m.match_data(pts[:0], start, 5)
    assert np.array_equal(est0, start)


def test_hector_just_once_semantics(pkg):
    """updateByScanJustOnce (OccGridMapBase.h:175-217): begin = cell (800, 800) whatever the pose; end = begin +
    round(p / 0.05); one beam along +x frees cells 800..end-1 and occupies the end cell."""
    m = port.PortHectorMap(1601, 1601, 0.05)
    visits = m.update_by_scan_just_once(np.array([[1.0, 0.0], [0.0, -0.524]], np.float32), (0.0, 0.0))
    lo, ui = m.cells()
    assert visits == (20 + 1) + (10 + 1)           # round(0.524 / 0.05) = round(10.48) = 10
    assert (ui[800, 800:820] == 1).all() and ui[800, 820] == 2
    assert (lo[800, 800:820] < 0).all() and lo[800, 820] > 0
    assert ui[790, 800] == 2 and (ui[791:800, 800] == 1).all()
    m.close()
