"""GPU tests of the lesson6 front end through the C ABI (b2s_mapper_*): every MatchScan on the CUDA matcher, near-chain
and loop-candidate matches batched.  Checked against the reference Mapper's golden output (tests/golden/karto_mapper.npz)
and against the reference Mapper with the same back end plugged in (its recorded answers where the reference build is
absent: tests/reference_replay.py)."""
import os

import numpy as np
import pytest

from oracle import ref
import mapper_cases as mc

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_mapper_cuda_vs_reference_golden(pkg):
    MP, abi = pkg.load("mapper"), pkg.abi
    assert pkg.load("matcher").device_count() > 0
    g = np.load(os.path.join(G, "karto_mapper.npz"))
    laser, prm, true, odom, ranges = mc.workload(pkg, int(g["seed"]), int(g["n"]))
    assert np.array_equal(ranges[::17], g["ranges_sample"])
    m = MP.Mapper(prm, abi.laser_from(laser))
    flags, _ = mc.run(m, odom, ranges)
    assert np.array_equal(flags, g["flags"])
    assert np.abs(m.poses() - g["poses"]).max() <= 1e-4            # contract; observed ~1e-12
    ids, diff, cov = m.edges()
    assert np.array_equal(ids, g["edge_ids"])                      # the same graph, edge for edge
    assert np.abs(diff - g["edge_diff"]).max() <= 1e-4 and np.abs(cov - g["edge_cov"]).max() <= 1e-4
    st = m.stats()
    assert st["loops_closed"] >= 1 and st["batches"] < st["match_calls"]
    print("mapper pose max |delta| vs reference:", np.abs(m.poses() - g["poses"]).max())
    m.close()


def test_mapper_cuda_multi_robot_vs_reference_golden(pkg):
    """Three robots into one mapper (b2s_mapper_process_sensor), every MatchScan on the CUDA matcher — the first-scan
    matches against another robot's whole scan list included — against the reference's three-sensor run."""
    MP, abi = pkg.load("mapper"), pkg.abi
    g = np.load(os.path.join(G, "karto_mapper_fleet.npz"))
    laser, prm, true, odom, ranges = mc.workload(pkg, int(g["seed"]), int(g["n"]), drift=mc.FLEET_DRIFT)
    assert np.array_equal(ranges[::17], g["ranges_sample"])
    m = MP.Mapper(prm, abi.laser_from(laser))
    flags, _ = mc.run_fleet(m, [None, "a_robot", "z_robot"], odom, ranges)
    assert np.array_equal(flags, g["flags"]) and np.abs(m.poses() - g["poses"]).max() <= 1e-4
    ids, diff, cov = m.edges()
    assert np.array_equal(ids, g["edge_ids"])
    assert np.abs(diff - g["edge_diff"]).max() <= 1e-4 and np.abs(cov - g["edge_cov"]).max() <= 1e-4
    sens = m.scan_sensors()
    assert (sens[ids[:, 0]] != sens[ids[:, 1]]).sum() >= 2 and m.stats()["loops_closed"] >= 1
    print("fleet pose max |delta| vs reference:", np.abs(m.poses() - g["poses"]).max())
    m.close()


def test_mapper_cuda_vs_live_reference_with_back_end(pkg, reference):
    MP, abi = pkg.load("mapper"), pkg.abi
    laser, prm, true, odom, ranges = mc.workload(pkg, 5, 130, drift=(0.01, 0.008, 0.004))
    g1, g2 = reference.new(MP.PoseGraph), MP.PoseGraph()
    r = reference.new(ref.RefMapper, prm, laser)
    r.set_scan_solver(g1.as_scan_solver())
    m = MP.Mapper(prm, abi.laser_from(laser))
    m.set_scan_solver(g2.as_scan_solver())
    for i in range(len(ranges)):
        a, b = r.process(ranges[i], odom[i], 0.1 * i), m.process(ranges[i], odom[i], 0.1 * i)
        assert a[0] == b[0] and np.abs(a[1] - b[1]).max() <= 1e-4, i
    assert np.abs(r.poses() - m.poses()).max() <= 1e-4
    assert np.array_equal(r.edges()[0], m.edges()[0])
    assert m.stats()["loops_closed"] >= 1 and g2.stats()["chi2_after"] < g2.stats()["chi2_before"]
    r.close(), m.close()


def test_mapper_default_parameters_run(pkg):
    """Mapper::InitializeParameters defaults (0.3 m / 0.01 m sequential window on a 2431^2 grid, 8 m / 0.05 m loop window,
    70-scan running buffer): a short stream must run and stay close to the truth."""
    MP, abi = pkg.load("mapper"), pkg.abi
    laser = pkg.synth.Laser()
    world, true, odom, ranges = pkg.synth.make_loop_trajectory(11, 30, laser, radius=2.0, step=0.25)
    m = MP.Mapper(MP.default_params(laser.range_threshold), abi.laser_from(laser))
    flags, _ = mc.run(m, odom, ranges)
    assert flags.all() and np.abs(m.poses()[:, :2] - true[:, :2]).max() < 0.05
    m.close()
