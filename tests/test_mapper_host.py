"""CPU tests of the mapper's HOST logic (karto_mapper.cu: key-frame gate, running window, graph edges, near chains,
loop-closure candidates, ScanSolver plug-in) against the UNMODIFIED reference karto::Mapper (oracle/_ref/libkarto_ref.so,
or its recorded answers where that build is absent: tests/reference_replay.py).
No GPU here: the product's matcher plug-in point is served by the CPU restatement's MatchScan (tests only), the
reference uses its own ScanMatcher — so every difference would come from the graph / pose logic under test."""
import os

import numpy as np
import pytest

from oracle import port, ref
import mapper_cases as mc

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def compare(r, m, tol=1e-9):
    pr, pm = r.poses(), m.poses()
    assert pr.shape == pm.shape and np.abs(pr - pm).max() <= tol
    (ir, dr, cr), (im, dm, cm) = r.edges(), m.edges()
    assert np.array_equal(ir, im), "graph edges differ"
    assert np.abs(dr - dm).max() <= tol and np.abs(cr - cm).max() <= tol


def test_mapper_matches_reference_without_back_end(pkg, reference):
    """150 scans, 3 laps: sequential matches against the running window, near-chain links (batched), loop closures
    accepted without a solver (the lesson6 indoor yaml: use_back_end false)."""
    MP, abi = pkg.load("mapper"), pkg.abi
    laser, prm, true, odom, ranges = mc.workload(pkg, 3, 150)
    al = abi.laser_from(laser)
    r = reference.new(ref.RefMapper, prm, laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    fr, cr = mc.run(r, odom, ranges)
    fm, cm = mc.run(m, odom, ranges)
    assert np.array_equal(fr, fm) and fr.all() and np.abs(cr - cm).max() <= 1e-9
    compare(r, m)
    st = m.stats()
    assert st["loops_closed"] >= 1 and st["running_scans"] == r.running_count() == 20
    assert st["batches"] < st["match_calls"]  # near chains / candidates went out batched
    ids = m.edges()[0]
    assert (ids[:, 1] - ids[:, 0] > 30).any()  # links across laps exist
    assert np.abs(m.poses()[:, :2] - true[:, :2]).max() < np.abs(odom[:, :2] - true[:, :2]).max()
    r.close(), m.close()


def test_mapper_with_scan_solver_plugin(pkg, reference):
    """The same back end (the library's pose-graph optimiser, one instance per side) plugged into the reference Mapper
    through karto::ScanSolver and into ours through b2s_scan_solver: corrected poses agree after every loop closure."""
    MP, abi = pkg.load("mapper"), pkg.abi
    laser, prm, true, odom, ranges = mc.workload(pkg, 5, 130, drift=(0.01, 0.008, 0.004))
    al = abi.laser_from(laser)
    g1, g2 = reference.new(MP.PoseGraph), MP.PoseGraph()
    r = reference.new(ref.RefMapper, prm, laser)
    r.set_scan_solver(g1.as_scan_solver())
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    m.set_scan_solver(g2.as_scan_solver())
    for i in range(len(ranges)):
        a, b = r.process(ranges[i], odom[i], 0.1 * i), m.process(ranges[i], odom[i], 0.1 * i)
        assert a[0] == b[0] and np.abs(a[1] - b[1]).max() <= 1e-9, i
    compare(r, m)
    s1, s2 = g1.stats(), g2.stats()
    assert s1 == s2 and s2["constraints"] == len(m.edges()[0]) and s2["chi2_after"] < 0.5 * s2["chi2_before"]
    assert m.stats()["loops_closed"] >= 1
    assert np.abs(m.poses()[:, :2] - true[:, :2]).max() < 0.5 * np.abs(odom[:, :2] - true[:, :2]).max()
    r.close(), m.close()


def test_mapper_key_frame_gate(pkg, reference):
    """Mapper::HasMovedEnough (Mapper.cpp:2087-2119): travel distance, heading and time interval."""
    MP, abi = pkg.load("mapper"), pkg.abi
    laser, prm, true, odom, ranges = mc.workload(pkg, 7, 12)
    prm.minimum_time_interval = 5.0
    al = abi.laser_from(laser)
    r = reference.new(ref.RefMapper, prm, laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    seq = [(0, 0.0), (0, 1.0), (1, 2.0), (1, 3.0), (1, 9.0), (2, 9.5)]  # (pose index, time): repeats are rejected
    tiny = odom[2] + np.array([0.05, 0.0, 0.02])
    for k, (i, t) in enumerate(seq):
        a, b = r.process(ranges[i], odom[i], t), m.process(ranges[i], odom[i], t)
        assert a[0] == b[0] and np.abs(a[1] - b[1]).max() <= 1e-9, k
    a, b = r.process(ranges[2], tiny, 10.0), m.process(ranges[2], tiny, 10.0)  # moved 5 cm / 0.02 rad: rejected
    assert a[0] == b[0] == False and np.abs(a[1] - b[1]).max() <= 1e-9
    turn = odom[2] + np.array([0.0, 0.0, 0.2])
    a, b = r.process(ranges[2], turn, 10.5), m.process(ranges[2], turn, 10.5)  # turned 0.2 rad >= 10 deg: accepted
    assert a[0] == b[0] == True
    assert len(m.poses()) == len(r.poses()) == 5
    compare(r, m)
    r.close(), m.close()


@pytest.mark.parametrize("prefixes,solver,seed", [(("a_robot", "z_robot"), False, 3), (("z_robot", "a_robot"), True, 7)])
def test_mapper_multi_robot_matches_reference(pkg, reference, prefixes, solver, seed):
    """MapperSensorManager semantics with three sensors (Mapper.cpp:45-100, 920-952, 1170-1275, 1333-1394, 2063-2070):
    a sensor's first scan is matched against all scans of the other sensors and linked to their first scans, near
    chains follow the near scan's own sensor, loop closures are searched per sensor in NAME order — the two extra
    robots' names sort before / after the first one's in both permutations."""
    MP, abi = pkg.load("mapper"), pkg.abi
    laser, prm, true, odom, ranges = mc.workload(pkg, seed, 150, drift=mc.FLEET_DRIFT)
    al = abi.laser_from(laser)
    r = reference.new(ref.RefMapper, prm, laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    if solver:
        g1, g2 = reference.new(MP.PoseGraph), MP.PoseGraph()
        r.set_scan_solver(g1.as_scan_solver())
        m.set_scan_solver(g2.as_scan_solver())
    ref_ids = [0] + [r.add_sensor(p) for p in prefixes]
    names = [None] + list(prefixes)  # None = b2s_mapper_process = the sensor "laser" ("a_robot" < "laser" < "z_robot")
    for k, (rob, i) in enumerate(mc.fleet_events()):
        a = r.process(ranges[i], odom[i], 0.1 * k, sensor=ref_ids[rob])
        b = m.process(ranges[i], odom[i], 0.1 * k, sensor=names[rob])
        assert a[0] == b[0] and np.abs(a[1] - b[1]).max() <= 1e-9, (k, rob, i)
    pr, pm = r.poses_by_id(), m.poses()
    assert pr.shape == pm.shape == (150, 3) and np.abs(pr - pm).max() <= 1e-9
    (ir, dr, cr), (im, dm, cm) = r.edges(), m.edges()
    assert np.array_equal(ir, im), "graph edges differ"
    assert np.abs(dr - dm).max() <= 1e-9 and np.abs(cr - cm).max() <= 1e-9
    sens = m.scan_sensors()
    rank = {p: k for k, p in enumerate(sorted(["laser"] + list(prefixes)))}
    assert sens[0] == rank["laser"] and sens[8] == rank["laser"] and sens[9] == rank[prefixes[0]]
    # links between different robots exist (first-scan links and near chains), and some loop was examined
    cross = sens[im[:, 0]] != sens[im[:, 1]]
    assert cross.sum() >= 2
    first_b = np.flatnonzero(sens == rank[prefixes[0]])[0]
    assert any((s_ == 0 and d_ == first_b) for s_, d_ in im), "first scan of robot 2 is linked to the first scan of robot 1"
    assert m.stats()["loops_closed"] >= 1
    if solver:
        assert g1.stats() == g2.stats()
    r.close(), m.close()


def test_mapper_multi_robot_golden(pkg):
    """The three-robot run as the reference left it (tests/golden/make_golden.py fleet), wherever the library loads."""
    MP, abi = pkg.load("mapper"), pkg.abi
    g = np.load(os.path.join(G, "karto_mapper_fleet.npz"))
    laser, prm, true, odom, ranges = mc.workload(pkg, int(g["seed"]), int(g["n"]), drift=mc.FLEET_DRIFT)
    assert np.array_equal(ranges[::17], g["ranges_sample"]), "the synthetic workload changed: regenerate the golden file"
    al = abi.laser_from(laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    flags, _ = mc.run_fleet(m, [None, "a_robot", "z_robot"], odom, ranges)
    assert np.array_equal(flags, g["flags"]) and np.abs(m.poses() - g["poses"]).max() <= 1e-9
    ids, diff, cov = m.edges()
    assert np.array_equal(ids, g["edge_ids"]) and np.abs(diff - g["edge_diff"]).max() <= 1e-9
    assert np.abs(cov - g["edge_cov"]).max() <= 1e-9
    m.close()


def test_mapper_golden(pkg):
    """Poses and edges the reference Mapper produced for the seeded workload (tests/golden/make_golden.py mapper),
    checked wherever the library loads — e.g. on the GPU box, where /root/reference does not exist."""
    MP, abi = pkg.load("mapper"), pkg.abi
    g = np.load(os.path.join(G, "karto_mapper.npz"))
    laser, prm, true, odom, ranges = mc.workload(pkg, int(g["seed"]), int(g["n"]))
    assert np.array_equal(ranges[::17], g["ranges_sample"]), "the synthetic workload changed: regenerate the golden file"
    al = abi.laser_from(laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    flags, _ = mc.run(m, odom, ranges)
    assert np.array_equal(flags, g["flags"])
    assert np.abs(m.poses() - g["poses"]).max() <= 1e-9
    ids, diff, cov = m.edges()
    assert np.array_equal(ids, g["edge_ids"]) and np.abs(diff - g["edge_diff"]).max() <= 1e-9
    assert np.abs(cov - g["edge_cov"]).max() <= 1e-9
    m.close()


def test_pose_graph_solver_recovers_ring(pkg):
    """The back-end optimiser on its own: a ring of 40 poses with exact relative constraints and a corrupted initial
    guess converges back to the ring (chi^2 -> 0) with the first node fixed."""
    import ctypes as C
    MP = pkg.load("mapper")
    n = 40
    th = np.arange(n) * 2 * np.pi / n
    truth = np.stack([3 * np.cos(th), 3 * np.sin(th), (th + np.pi / 2 + np.pi) % (2 * np.pi) - np.pi], 1)
    rng = np.random.default_rng(1)
    guess = truth + np.concatenate([np.zeros((1, 3)), rng.normal(0, [0.2, 0.2, 0.1], (n - 1, 3))])
    g = MP.PoseGraph()
    s = g.as_scan_solver()
    for i in range(n):
        s.add_node(s.user, i, guess[i].ctypes.data_as(C.POINTER(C.c_double)))
    cov = (np.eye(3) * [1e-3, 1e-3, 1e-4]).ravel()
    for i in range(n):
        for j in ((i + 1) % n, (i + 3) % n):
            a, b = truth[i], truth[j]
            c, sn = np.cos(a[2]), np.sin(a[2])
            d = np.array([c * (b[0] - a[0]) + sn * (b[1] - a[1]), -sn * (b[0] - a[0]) + c * (b[1] - a[1]),
                          (b[2] - a[2] + np.pi) % (2 * np.pi) - np.pi])
            s.add_constraint(s.user, i, j, d.ctypes.data_as(C.POINTER(C.c_double)), cov.ctypes.data_as(C.POINTER(C.c_double)))
    ids, poses = np.zeros(n, np.int32), np.zeros((n, 3))
    got = s.compute(s.user, n, ids.ctypes.data_as(C.POINTER(C.c_int32)), poses.ctypes.data_as(C.POINTER(C.c_double)))
    st = g.stats()
    assert got == n and list(ids) == list(range(n))
    assert st["chi2_after"] < 1e-12 * max(1.0, st["chi2_before"]) and st["chi2_before"] > 100
    d = poses - truth
    d[:, 2] = (d[:, 2] + np.pi) % (2 * np.pi) - np.pi
    assert np.abs(d).max() < 1e-6
    g.close()


def test_pose_graph_sparse_ldlt_reaches_the_least_squares_optimum(pkg):
    """The sparse block LDL^T back end on a noisy multi-lap graph with loop closures (fill-in exercised: the minimum-degree
    order has to eliminate through the loop edges): its final chi^2 equals the optimum scipy's trust-region least-squares
    solver finds from the same start, and the poses agree to 1e-5."""
    import ctypes as C
    from scipy.optimize import least_squares
    MP = pkg.load("mapper")
    n, per_lap = 160, 40
    th = np.arange(n) * 2 * np.pi / per_lap
    truth = np.stack([4 * np.cos(th), 4 * np.sin(th), (th + np.pi / 2 + np.pi) % (2 * np.pi) - np.pi], 1)
    rng = np.random.default_rng(7)

    def rel(a, b):
        c, sn = np.cos(a[2]), np.sin(a[2])
        return np.array([c * (b[0] - a[0]) + sn * (b[1] - a[1]), -sn * (b[0] - a[0]) + c * (b[1] - a[1]),
                         (b[2] - a[2] + np.pi) % (2 * np.pi) - np.pi])
    guess = truth + np.concatenate([np.zeros((1, 3)), rng.normal(0, [0.05, 0.05, 0.02], (n - 1, 3))])
    sig = np.array([0.02, 0.02, 0.005])
    cons = []
    for i in range(n):
        for j in [i + 1, i + 2] + ([i - per_lap] if i >= per_lap and i % 3 == 0 else []):
            if 0 <= j < n and j != i:
                a, b = (i, j) if j > i else (j, i)
                cons.append((a, b, rel(truth[a], truth[b]) + rng.normal(0, sig)))
    g = MP.PoseGraph()
    s = g.as_scan_solver()
    dp = C.POINTER(C.c_double)
    for i in range(n):
        s.add_node(s.user, i, np.ascontiguousarray(guess[i]).ctypes.data_as(dp))
    cov = np.ascontiguousarray(np.diag(sig ** 2).ravel())
    for a, b, d in cons:
        s.add_constraint(s.user, a, b, np.ascontiguousarray(d).ctypes.data_as(dp), cov.ctypes.data_as(dp))
    ids, poses = np.zeros(n, np.int32), np.zeros((n, 3))
    assert s.compute(s.user, n, ids.ctypes.data_as(C.POINTER(C.c_int32)), poses.ctypes.data_as(dp)) == n
    st = g.stats()

    def residuals(x):
        P = np.concatenate([guess[:1], x.reshape(-1, 3)])
        out = []
        for a, b, d in cons:
            e = rel(P[a], P[b]) - d
            e[2] = (e[2] + np.pi) % (2 * np.pi) - np.pi
            out.append(e / sig)
        return np.concatenate(out)
    opt = least_squares(residuals, guess[1:].ravel(), method="trf", xtol=1e-14, ftol=1e-14, gtol=1e-12)
    chi_opt = float((opt.fun ** 2).sum())
    assert st["chi2_after"] <= chi_opt * (1 + 1e-6) and st["chi2_after"] < 0.5 * st["chi2_before"]
    d = poses[1:] - opt.x.reshape(-1, 3)
    d[:, 2] = (d[:, 2] + np.pi) % (2 * np.pi) - np.pi
    assert np.abs(d).max() < 1e-5
    g.close()


def test_mapper_with_dropouts(pkg, reference):
    """1 % of the readings replaced by NaN / 0.0 (below min range): unfiltered points, barycenters and every decision
    still agree with the reference exactly."""
    MP, abi = pkg.load("mapper"), pkg.abi
    laser, prm, true, odom, ranges = mc.workload(pkg, 3, 70)
    rng = np.random.default_rng(4)
    r2 = ranges.copy()
    for k, (i, j) in enumerate(np.argwhere(rng.random(r2.shape) < 0.01)):
        r2[i, j] = np.nan if k % 2 == 0 else 0.0
    al = abi.laser_from(laser)
    r = reference.new(ref.RefMapper, prm, laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    fr, _ = mc.run(r, odom, r2)
    fm, _ = mc.run(m, odom, r2)
    assert np.array_equal(fr, fm)
    compare(r, m)
    r.close(), m.close()


def test_mapper_singular_covariance_is_an_error_where_the_reference_asserts(pkg, reference, tmp_path):
    """ComputeWeightedMean inverts the link covariances with Matrix3::Inverse, which ASSERTS when |det| <= 1e-14
    (Karto.h:2445-2453; the catkin build keeps asserts).  On this seeded stream the reference aborts at some scan; ours
    must report B2S_ERR_BAD_STATE at the same scan instead of continuing with garbage."""
    import subprocess
    import sys
    MP, abi = pkg.load("mapper"), pkg.abi
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import importlib, mapper_cases as mc\nfrom oracle import ref\n"
            "pkg = importlib.import_module('creating-2d-laser-slam-from-scratch_b200')\n"
            "laser, prm, true, odom, ranges = mc.workload(pkg, 9, 70)\nr = ref.RefMapper(prm, laser)\n"
            "for i in range(70):\n    print(i, flush=True)\n    r.process(ranges[i], odom[i], 0.1 * i)\nprint('done', flush=True)\n"
            % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__))))
    laser, prm, true, odom, ranges = mc.workload(pkg, 9, 70)

    def reference_failing_scan(*workload):  # runs `code`; the workload is passed to tie the recording to it
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
        lines = out.stdout.split()
        assert out.returncode != 0 and lines[-1] != "done" and "Assertion" in out.stderr
        return int(lines[-1])
    ref_fail = reference.call("scan at which the reference Mapper asserts", reference_failing_scan, prm, laser, odom, ranges)
    al = abi.laser_from(laser)
    m = MP.Mapper(prm, al, match_fn=port.mapper_match_hook(prm, al))
    ours_fail = None
    for i in range(70):
        try:
            m.process(ranges[i], odom[i], 0.1 * i)
        except pkg.load("matcher").B2SError as e:
            assert e.status == abi.B2S_ERR_BAD_STATE
            ours_fail = i
            break
    assert ours_fail == ref_fail
    m.close()


def test_mapper_default_params_equal_the_reference(pkg, reference):
    """b2s_mapper_default_params vs the values a fresh karto::Mapper holds (Mapper::InitializeParameters)."""
    import ctypes as C
    MP = pkg.load("mapper")
    ours = MP.default_params(12.0)

    def reference_defaults():
        theirs = MP.MapperParams()
        ref._lib(False).ref_mapper_default_params(C.byref(theirs))
        theirs.sequential.range_threshold = theirs.loop.range_threshold = 12.0  # comes from the laser, not the Mapper
        return flat(theirs)

    def flat(p):
        out = {}
        for name, _ in p._fields_:
            v = getattr(p, name)
            if hasattr(v, "_fields_"):
                out.update({f"{name}.{k}": getattr(v, k) for k, _ in v._fields_})
            else:
                out[name] = v
        return out
    a, b = flat(ours), reference.call("karto::Mapper default parameters", reference_defaults)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k] == b[k], (k, a[k], b[k])
