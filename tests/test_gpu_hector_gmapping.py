"""GPU parity tests for K2a (Hector log-odds update), K3 (Hector Gauss-Newton) and K2b (GMapping counters) through
the C ABI.  Gates: traversed cells / update indices / integer counters bit-exact; log-odds floats bit-exact (same
float32 operations in the reference's order); the HectorSlamProcessor's Gauss-Newton poses / Hessians bit-exact in its
default exact mode (1e-4 in fast mode; the single-level b2s_hector_map_match_data keeps 1e-4); GMapping acc floats within
float rounding.
The Hector restatement is itself pinned bit for bit to the reference headers (tests/test_oracle_hector_reference.py);
where the reference build travelled with the repo (oracle/_ref/libhector_ref.so) the CUDA path is compared with it directly."""
import os

import numpy as np
import pytest

from oracle import port

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def mods(pkg):
    assert pkg.load("matcher").device_count() > 0
    return pkg.load("hector"), pkg.load("gmapping")


def test_hector_update_stream(pkg, mods):
    """60-scan trajectory into a 1024^2 map (node settings: update factors 0.4 / 0.9), cell-for-cell identical
    log-odds and update indices after every 10th scan, incl. the <50 clamp region after repeated hits."""
    H, _ = mods
    laser = pkg.synth.Laser()
    world, poses, ranges = pkg.synth.make_trajectory(4, 60, laser, step_xy=0.1, step_th_deg=3)
    g, c = H.HectorMap(1024, 1024, 0.05), port.PortHectorMap(1024, 1024, 0.05)
    g.set_factors(0.4, 0.9)
    c.set_factors(0.4, 0.9)
    for i in range(60):
        pts = H.scan_to_data_container(ranges[i], laser, 0.05)
        wp = poses[i].astype(np.float32)
        for _ in range(1 if i < 50 else 4):  # hammer the last poses to reach the clamp
            g.update_by_scan(pts, (0.0, 0.0), wp)
            c.update_by_scan(pts, (0.0, 0.0), wp)
        if i % 10 == 9:
            (glo, gui), (clo, cui) = g.cells(), c.cells()
            assert np.array_equal(gui, cui)
            assert np.array_equal(glo, clo)
    assert glo.max() >= 50.0
    ros = g.ros_map()
    assert ((ros == 0) == (clo < 0)).all() and ((ros == 100) == (clo > 0)).all() and ((ros == -1) == (clo == 0)).all()
    assert g.last_timing()["update_ms"] > 0


def test_hector_origo_offset_and_out_of_map(pkg, mods):
    H, _ = mods
    laser = pkg.synth.Laser()
    mc = pkg.synth.make_match_case(9)
    pts = H.scan_to_data_container(mc.ranges, laser, 0.1)
    for size, start in ((256, (0.5, 0.5)), (128, (0.3, 0.7)), (64, (0.5, 0.5))):  # small maps: many beams leave the map
        g, c = H.HectorMap(size, size, 0.1, *start), port.PortHectorMap(size, size, 0.1, *start)
        wp = np.array([0.7, -0.4, 2.1], np.float32)
        g.update_by_scan(pts, (2.0, -1.5), wp)
        c.update_by_scan(pts, (2.0, -1.5), wp)
        assert np.array_equal(g.cells()[0], c.cells()[0]) and np.array_equal(g.cells()[1], c.cells()[1])


def test_hector_update_by_scan_just_once(pkg, mods):
    """The lesson4 make-map demo variant (OccGridMapBase.h:175-217): 1600^2 map (the fixed map pose is cell 800, 800),
    points in metres with half-cell values (round half away from zero), repeated scans, origo offset."""
    H, _ = mods
    laser = pkg.synth.Laser()
    g, c = H.HectorMap(1601, 1601, 0.05), port.PortHectorMap(1601, 1601, 0.05)
    for seed, origo in ((11, (0.0, 0.0)), (12, (0.0, 0.0)), (13, (3.2, -1.7)), (11, (0.0, 0.0))):
        mc = pkg.synth.make_match_case(seed)
        th = laser.min_angle + laser.angular_resolution * np.arange(laser.n_readings)
        r = np.where(np.isfinite(mc.ranges), mc.ranges, 0.0)
        pts = np.stack([r * np.cos(th), r * np.sin(th)], axis=1).astype(np.float32)
        pts[::7] = np.round(pts[::7] / 0.05) * 0.05 + 0.025  # exact .5 cells: ::round semantics
        pts[5] = (1000.0, 3.0)  # leaves the map: skipped
        g.update_by_scan_just_once(pts, origo)
        c.update_by_scan_just_once(pts, origo)
        (glo, gui), (clo, cui) = g.cells(), c.cells()
        assert np.array_equal(gui, cui)
        assert np.array_equal(glo, clo)
    assert (gui >= 0).sum() > 10000


def test_hector_match_data(pkg, mods):
    """K3: three pyramid levels like MapRepMultiMap::matchData (3 / 3 / 5 extra iterations), level by level."""
    H, _ = mods
    laser = pkg.synth.Laser()
    world, poses, ranges = pkg.synth.make_trajectory(6, 12, laser, step_xy=0.08, step_th_deg=2)
    levels = [(1024, 0.05), (512, 0.1), (256, 0.2)]
    gm = [H.HectorMap(s, s, r) for s, r in levels]
    cm = [port.PortHectorMap(s, s, r) for s, r in levels]
    for m in gm + cm:
        m.set_factors(0.4, 0.9)
    for i in range(11):
        for (s, r), g, c in zip(levels, gm, cm):
            pts = H.scan_to_data_container(ranges[i], laser, r)
            g.update_by_scan(pts, (0, 0), poses[i].astype(np.float32))
            c.update_by_scan(pts, (0, 0), poses[i].astype(np.float32))
    est_g = est_c = (poses[10] + np.array([0.04, -0.03, 0.02])).astype(np.float32)
    for lvl in (2, 1, 0):
        pts = H.scan_to_data_container(ranges[11], laser, levels[lvl][1])
        est_g, cov_g = gm[lvl].match_data(pts, est_g, 5 if lvl == 0 else 3)
        est_c, cov_c = cm[lvl].match_data(pts, est_c, 5 if lvl == 0 else 3)
        assert np.allclose(est_g, est_c, rtol=0, atol=1e-4), (lvl, est_g, est_c)
        assert np.allclose(cov_g, cov_c, rtol=1e-3, atol=1e-2)
    assert np.abs(est_g[:2] - poses[11][:2]).max() < 0.05
    assert gm[0].last_timing()["match_ms"] > 0
    e, _ = gm[0].match_data(np.zeros((0, 2), np.float32), est_g, 5)
    assert np.array_equal(e, est_g)


def _cell_mismatch(a, b):
    (la, ua), (lb, ub) = a, b
    touched = (ua >= 0) | (ub >= 0)
    return int(((ua != ub) | (la.view(np.int32) != lb.view(np.int32)))[touched].sum()), int(touched.sum())


def _processors(kw):
    """CPU side of the processor tests: the restatement always, the reference build itself where it is present."""
    from oracle import ref_hector as rh
    out = [("restatement", port.PortHectorProcessor(**kw))]
    if rh.available():
        out.append(("reference", rh.RefHectorProcessor(**kw)))
    return out


def test_hector_slam_given_poses_bit_exact(pkg, mods):
    """HectorSlamProcessor::update(map_without_matching=true) with the poses given: all three pyramid levels equal the
    CPU processor's cell for cell (float32 log-odds bit patterns and update indices) — including the reference's stale
    coarse-level containers (levels > 0 reuse the last MATCHED scan) and the map-update gate."""
    H, _ = mods
    laser = pkg.synth.Laser()
    _, poses, ranges = pkg.synth.make_trajectory(8, 40, laser, step_xy=0.1, step_th_deg=3)
    kw = dict(resolution=0.05, size_x=1000, size_y=1000, start=(0.5, 0.5), levels=3, min_dist=0.2, min_angle=0.1)
    g = H.HectorSlam(**kw)
    cpus = _processors(kw)
    for i in range(40):
        pts = H.scan_to_data_container(ranges[i], laser, 0.05)
        wp = poses[i].astype(np.float32)
        without = i % 3 != 1  # every third scan is matched from the true pose (fills the coarse containers)
        eg, _ = g.update(pts, (0.1, -0.2), wp, without)
        for name, c in cpus:
            ec, _ = c.update(pts, (0.1, -0.2), wp, without)
            if without:
                assert np.array_equal(eg, ec) and np.array_equal(eg, wp), name
            else:  # matched scans: the device's Gauss-Newton pose is the CPU's, bit for bit (exact mode)
                assert np.array_equal(eg.view(np.int32), ec.view(np.int32)), (name, i, eg, ec)
    st = g.stats()
    assert st["updated"] >= 27 and st["cell_visits"] > 1_000_000
    for name, c in cpus:
        for lvl in range(3):
            bad, touched = _cell_mismatch(g.level(lvl), c.level(lvl))
            assert touched > 1000 and bad == 0, (name, lvl, bad, touched)
    ros = g.ros_map(0)
    lo0 = g.level(0)[0]
    assert ((ros == 0) == (lo0 < 0)).all() and ((ros == 100) == (lo0 > 0)).all()


def test_hector_slam_mapping_only_bit_exact(pkg, mods):
    """Pure mapping (every scan map_without_matching): no device transcendental touches the integer path, so level 0 is
    bit-identical; levels > 0 never receive data (the reference only fills dataContainers in matchData)."""
    H, _ = mods
    laser = pkg.synth.Laser()
    _, poses, ranges = pkg.synth.make_trajectory(9, 30, laser, step_xy=0.1, step_th_deg=3)
    kw = dict(resolution=0.05, size_x=1024, size_y=1024, start=(0.4, 0.6), levels=3)
    g = H.HectorSlam(**kw)
    cpus = _processors(kw)
    for i in range(30):
        pts = H.scan_to_data_container(ranges[i], laser, 0.05)
        for _ in range(1 if i < 25 else 5):  # reach the <50 clamp
            g.update(pts, (0, 0), poses[i].astype(np.float32), True)
            for _, c in cpus:
                c.update(pts, (0, 0), poses[i].astype(np.float32), True)
    for name, c in cpus:
        for lvl in range(3):
            (gl, gu), (cl, cu) = g.level(lvl), c.level(lvl)
            assert np.array_equal(gu, cu) and np.array_equal(gl.view(np.int32), cl.view(np.int32)), (name, lvl)
    assert g.level(0)[0].max() >= 50.0 and (g.level(1)[1] >= 0).sum() == 0
    g.reset()
    assert (g.level(0)[1] == -1).all() and (g.level(0)[0] == 0).all()


def test_hector_slam_stream_and_golden(pkg, mods):
    """Self-driven SLAM stream (hint = previous estimate, as the node runs): the pose / Hessian trace EQUALS the
    reference's golden trace (tests/golden/hector.npz, produced by the reference headers) bit for bit and so do the maps."""
    H, _ = mods
    g = np.load(os.path.join(G, "hector.npz"))
    kw = dict(resolution=float(g["resolution"]), size_x=int(g["size"]), size_y=int(g["size"]), start=(0.5, 0.5), levels=3,
              min_dist=float(g["min_dist"]), min_angle=float(g["min_angle"]))
    p = H.HectorSlam(**kw)
    est = g["start_pose"].astype(np.float32)
    for i in range(int(g["n_scans"])):
        est, cov = p.update(g[f"pts{i}"], (0, 0), est, bool(g["without_matching"][i]))
        ref_pose, ref_cov = g["trace"][i][:3], g["trace"][i][3:].reshape(3, 3)
        assert np.array_equal(est.view(np.int32), ref_pose.view(np.int32)), (i, est, ref_pose)
        if not g["without_matching"][i]:
            assert np.array_equal(cov.view(np.int32), ref_cov.view(np.int32)), i
    for lvl in range(3):
        lo, ui = p.level(lvl)
        ref_ui = np.full(ui.size, -1, np.int32)
        ref_lo = np.zeros(ui.size, np.float32)
        ref_ui[g[f"l{lvl}_idx"]] = g[f"l{lvl}_ui"]
        ref_lo[g[f"l{lvl}_idx"]] = g[f"l{lvl}_lo"]
        bad, touched = _cell_mismatch((lo.ravel(), ui.ravel()), (ref_lo, ref_ui))
        assert touched > 500 and bad == 0, (lvl, bad, touched)


def _stream_case(pkg, H, seed, n, step_xy=0.05, step_th=1.5):
    laser = pkg.synth.Laser()
    _, poses, ranges = pkg.synth.make_trajectory(seed, n, laser, step_xy=step_xy, step_th_deg=step_th)
    return poses, [H.scan_to_data_container(ranges[i], laser, 0.05) for i in range(n)]


def test_hector_slam_self_driven_stream_bit_exact(pkg, mods):
    """The node's loop (hint = last scan-match pose) over 120 scans with the node defaults: every pose, every gate
    decision and all three maps equal the CPU processor's bit for bit; the one-call stream form gives the same again."""
    H, _ = mods
    poses, scans = _stream_case(pkg, H, 31, 120)
    kw = dict(resolution=0.05, size_x=1000, size_y=1000, start=(0.5, 0.5), levels=3, update_free=0.4, update_occupied=0.9,
              min_dist=0.08, min_angle=0.9)  # the synthetic walk drifts slowly: a low distance gate opens it a few times
    g, g2 = H.HectorSlam(**kw), H.HectorSlam(**kw)
    cpus = _processors(kw)
    est = poses[0].astype(np.float32)
    ests = {name: est.copy() for name, _ in cpus}
    trace, flags = [], []
    for i in range(len(scans)):
        est, cov = g.update(scans[i], (0, 0), est)
        trace.append(est.copy()); flags.append(g.map_updated)
        for name, c in cpus:
            ests[name], cc = c.update(scans[i], (0, 0), ests[name])
            assert np.array_equal(est.view(np.int32), ests[name].view(np.int32)), (name, i, est, ests[name])
            assert np.array_equal(cov.view(np.int32), cc.view(np.int32)), (name, i)
    assert 3 <= sum(flags) < len(scans)  # the gate opened a few times, not always
    assert np.abs(est[:2] - poses[-1][:2]).max() < 0.1
    p2, u2, cov2 = g2.process_stream(scans, (0, 0), first_hint=poses[0].astype(np.float32))
    assert np.array_equal(p2.view(np.int32), np.stack(trace).view(np.int32)) and list(u2) == flags
    assert np.array_equal(cov2.view(np.int32), cov.view(np.int32))
    a, u = g2.last_poses()
    assert np.array_equal(a, trace[-1])
    for lvl in range(3):
        for name, c in cpus:
            bad, touched = _cell_mismatch(g.level(lvl), c.level(lvl))
            assert touched > 1000 and bad == 0, (name, lvl, bad, touched)
        bad, _ = _cell_mismatch(g.level(lvl), g2.level(lvl))
        assert bad == 0
    st = g2.stats()
    assert st["matched"] == len(scans) and st["updated"] == sum(flags) and st["match_ms"] > 0


def test_hector_slam_fast_mode_within_contract(pkg, mods):
    """set_exact(0): tree-summed Gauss-Newton terms and device sinf/cosf/expf — poses within the 1e-4 contract of the
    CPU processor when both are fed the same hints; cells may differ where a pose moved by an ulp."""
    H, _ = mods
    poses, scans = _stream_case(pkg, H, 32, 40, step_xy=0.1, step_th=3)
    kw = dict(resolution=0.05, size_x=1000, size_y=1000, start=(0.5, 0.5), levels=3, min_dist=0.2, min_angle=0.1)
    g = H.HectorSlam(exact=False, **kw)
    c = port.PortHectorProcessor(**kw)
    for i in range(len(scans)):
        wp = poses[i].astype(np.float32)
        eg, _ = g.update(scans[i], (0, 0), wp)
        ec, _ = c.update(scans[i], (0, 0), wp)
        assert np.abs(eg - ec).max() <= 1e-4, (i, eg, ec)
    for lvl in range(3):
        bad, touched = _cell_mismatch(g.level(lvl), c.level(lvl))
        assert touched > 1000 and bad <= max(2, touched // 500), (lvl, bad, touched)


def test_hector_slam_fast_mode_cluster_match(pkg, mods):
    """Fast mode spreads the per-point phase of the match over a 4-CTA thread-block cluster (partial sums through
    distributed shared memory).  Same stream through the clustered kernel and the one-CTA fast match (a batched handle
    of one processor, hint = previous pose as the stream chains them): poses within the 1e-4 contract of each other and
    of the CPU processor, identical gate decisions; the clustered path is deterministic (per-scan calls and the one-call
    stream agree bit for bit)."""
    H, _ = mods
    poses, scans = _stream_case(pkg, H, 33, 60, step_xy=0.1, step_th=3)
    kw = dict(resolution=0.05, size_x=1000, size_y=1000, start=(0.5, 0.5), levels=3, min_dist=0.2, min_angle=0.1)
    first = poses[0].astype(np.float32)
    gc = H.HectorSlam(exact=False, **kw)
    if gc.cluster_size() != 4:  # (a device / driver that cannot co-schedule the cooperative grid as clusters: the handle
        pytest.skip("thread-block cluster launch not available here: the fast path runs on one CTA")  # falls back, see hs_create)
    pc, uc, _ = gc.process_stream(scans, (0, 0), first_hint=first)
    g1 = H.HectorSlam(exact=False, batch=1, **kw)
    est, p1, u1 = first[None], [], []
    for sc in scans:
        pb, _, ub = g1.update_batch([sc], (0, 0), est)
        est = pb.copy()
        p1.append(pb[0].copy()); u1.append(bool(ub[0]))
    p1 = np.stack(p1)
    c = port.PortHectorProcessor(**kw)
    est, ref_poses = first, []
    for sc in scans:
        est, _ = c.update(sc, (0, 0), est)
        ref_poses.append(est.copy())
    ref_poses = np.stack(ref_poses)
    assert np.abs(pc - p1).max() <= 1e-4 and np.abs(pc - ref_poses).max() <= 1e-4, (np.abs(pc - p1).max(), np.abs(pc - ref_poses).max())
    assert list(uc) == list(u1) and 2 <= sum(uc) < len(scans)
    g2 = H.HectorSlam(exact=False, **kw)
    est = first
    for i, sc in enumerate(scans):
        est, _ = g2.update(sc, (0, 0), est)
        assert np.array_equal(est.view(np.int32), pc[i].view(np.int32)), i
    for lvl in range(3):
        bad, touched = _cell_mismatch(gc.level(lvl), g2.level(lvl))
        assert touched > 1000 and bad == 0
    print("cluster vs one-CTA fast match: max |pose diff|", np.abs(pc - p1).max(), "vs CPU processor", np.abs(pc - ref_poses).max())


def test_hector_slam_batch_equals_single_processors(pkg, mods):
    """B = 3 independent processors behind one handle (different robots, ragged scans): each equals its own
    single-processor run bit for bit — poses, gate decisions, maps."""
    H, _ = mods
    kw = dict(resolution=0.05, size_x=512, size_y=512, start=(0.5, 0.5), levels=3, min_dist=0.3, min_angle=0.9)
    cases = [_stream_case(pkg, H, 40 + b, 25, step_xy=0.08, step_th=2) for b in range(3)]
    cases[1] = (cases[1][0], [s[::2] for s in cases[1][1]])  # a robot with half the beams
    cap = max(len(s) for _, sc in cases for s in sc)
    gb = H.HectorSlam(batch=3, max_points=cap, **kw)
    singles = [H.HectorSlam(**kw) for _ in range(3)]
    est = np.stack([c[0][0].astype(np.float32) for c in cases])
    for i in range(25):
        pb, cb, ub = gb.update_batch([cases[b][1][i] for b in range(3)], (0, 0), est)
        for b in range(3):
            e1, c1 = singles[b].update(cases[b][1][i], (0, 0), est[b])
            assert np.array_equal(pb[b].view(np.int32), e1.view(np.int32)), (i, b)
            assert np.array_equal(cb[b].view(np.int32), c1.view(np.int32)) and ub[b] == singles[b].map_updated
        est = pb.copy()
    for b in range(3):
        for lvl in range(3):
            bad, touched = _cell_mismatch(gb.level_of(b, lvl), singles[b].level(lvl))
            assert touched > 200 and bad == 0, (b, lvl)
    assert gb.stats()["matched"] == 75


def test_hector_slam_epoch_wrap(pkg, mods):
    """Per-scan stamps carry a 20-bit epoch: crossing it (stamps cleared, epochs restarted) changes nothing."""
    H, _ = mods
    poses, scans = _stream_case(pkg, H, 50, 12, step_xy=0.1, step_th=3)
    kw = dict(resolution=0.05, size_x=512, size_y=512, start=(0.5, 0.5), levels=2)
    g, c = H.HectorSlam(**kw), port.PortHectorProcessor(**kw)
    for i in range(12):
        if i == 3:
            g.debug_set_epoch((1 << 20) - 4)
        wp = poses[i].astype(np.float32)
        g.update(scans[i], (0, 0), wp, True)
        c.update(scans[i], (0, 0), wp, True)
    for lvl in range(2):
        bad, touched = _cell_mismatch(g.level(lvl), c.level(lvl))
        assert bad == 0 and (lvl > 0 or touched > 1000)


def test_gmapping_golden_and_oracle(pkg, mods):
    _, GM = mods
    g = np.load(os.path.join(G, "gmapping.npz"))
    for k in range(2):
        b = g[f"c{k}_bounds"]
        m = GM.GMap(*b)
        assert [m.size_x, m.size_y] == list(g[f"c{k}_size"])
        m.compute_map(g[f"c{k}_ranges"], g["angles"], tuple(g[f"c{k}_laser_xy"]))
        n, v, ax, ay = m.cells()
        ys, xs = np.nonzero(v)
        assert np.array_equal(np.stack([ys, xs], 1), g[f"c{k}_cells_yx"])
        assert np.array_equal(n[ys, xs], g[f"c{k}_n"]) and np.array_equal(v[ys, xs], g[f"c{k}_visits"])
        assert np.allclose(ax[ys, xs], g[f"c{k}_acc_x"], rtol=1e-6, atol=1e-5)
        assert np.allclose(ay[ys, xs], g[f"c{k}_acc_y"], rtol=1e-6, atol=1e-5)
        p = port.PortGMap(*b)
        p.compute_map(g[f"c{k}_ranges"], g["angles"], tuple(g[f"c{k}_laser_xy"]))
        assert np.array_equal(m.ros_map(), p.ros_map())
        m.close()


def test_gmapping_accumulate_and_errors(pkg, mods):
    _, GM = mods
    M = pkg.load("matcher")
    laser = pkg.synth.Laser()
    ang = (np.float32(laser.min_angle) + np.arange(1081, dtype=np.float32) * np.float32(laser.angular_resolution)).astype(np.float64)
    m, p = GM.GMap(-25, -25, 25, 25, 0.1), port.PortGMap(-25, -25, 25, 25, 0.1)
    for seed in range(6):
        r = pkg.synth.make_match_case(60 + seed, dropout=0.01).ranges.astype(np.float32).astype(np.float64)
        m.compute_map(r, ang, (0.3 * seed, -0.2 * seed))
        assert p.compute_map(r, ang, (0.3 * seed, -0.2 * seed)) == 0
    n, v, ax, ay = m.cells()
    pn, pv, pax, pay = p.cells()
    assert np.array_equal(n, pn) and np.array_equal(v, pv)
    assert np.allclose(ax, pax, rtol=1e-6, atol=1e-4) and np.allclose(ay, pay, rtol=1e-6, atol=1e-4)
    small = GM.GMap(-5, -5, 5, 5, 0.05)
    with pytest.raises(M.B2SError) as e:
        small.compute_map(np.full(1081, 20.0), ang)
    assert e.value.status == pkg.abi.B2S_ERR_OUT_OF_RANGE
    assert small.cells()[1].sum() == 0  # nothing was updated
