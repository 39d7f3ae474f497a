"""Angle pruning of the K1 window sweep (k_prune_select) against the dense sweep (kernel selector 3), per workload:
stage times (CUDA events, mean over the timed calls), the fraction of (match, angle) pairs swept, and whether the
outputs are identical.
  cfg2             : bench.py's headline batch (1024 seeded matches, one base scan each)
  running_window_70: grids rasterised from a 70-scan running window (the mapper's shape, 128 matches)
  empty_grids      : no base scans, every candidate ties: nothing can be pruned (worst-case cost of the bound pass)
usage: python tools/k1_prune_probe.py [out.json]"""
import importlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
pkg = importlib.import_module("creating-2d-laser-slam-from-scratch_b200")
abi, synth, M = pkg.abi, pkg.synth, pkg.load("matcher")
D = abi.KT_PI_180
params, laser = abi.matcher_params(1.5, 0.05, 0.03, 9.25), abi.laser_from(synth.Laser())
se = abi.Search(0.75, 0.75, 0.05, 0.05, 22.5 * D, 0.25 * D, 1, 0)


def cfg2(B=1024, base=1_000_000):
    cases = [synth.make_match_case(base + i) for i in range(B)]
    return (np.stack([c.ranges for c in cases]), np.stack([c.odom_pose for c in cases]),
            np.stack([c.base_ranges for c in cases])[:, None, :], np.stack([c.base_pose for c in cases])[:, None, :])


def running_window(nb=70, B=128):
    _, tp, tr = synth.make_trajectory(77, nb + 1, synth.Laser(), step_xy=0.1, step_th_deg=3)
    vr = np.tile(tr[-1][None], (B, 1))
    vp = np.tile(tp[-1][None], (B, 1)) + np.random.default_rng(1).uniform(-0.05, 0.05, (B, 3))
    return vr, vp, np.tile(tr[None, :nb], (B, 1, 1)), np.tile(tp[None, :nb], (B, 1, 1))


def empty(B=1024):
    r, p, _, _ = cfg2(B)
    return r, p, np.zeros((B, 0, r.shape[1])), np.zeros((B, 0, 3))


def measure(m, centers, kernel, calls=10):
    m.set_kernel(kernel)
    for _ in range(3):
        out = m.correlate_scan(centers, se)
    t = []
    for _ in range(calls):
        out = m.correlate_scan(centers, se)
        t.append(m.last_timing())
    row = {k: float(np.mean([x[k] for x in t])) for k in ("lut_ms", "sweep_ms", "reduce_ms")}
    row["step_ms"] = row["lut_ms"] + row["sweep_ms"] + row["reduce_ms"]
    row.update(m.last_prune_stats())
    m.set_kernel(0)
    return row, out


report = {}
for name, (r, p, br, bp) in (("cfg2", cfg2()), ("running_window_70", running_window()), ("empty_grids", empty())):
    B, nb = r.shape[0], max(br.shape[1], 1)
    m = M.ScanMatcher(params, laser, max_batch=B, max_base_scans=nb)
    m.set_scans(r, p)
    m.add_scans(br, bp)
    pruned, a = measure(m, p, 0)
    dense, b = measure(m, p, 3)
    report[name] = {"batch": B, "pruned": pruned, "dense": dense, "speedup": dense["step_ms"] / pruned["step_ms"],
                    "identical": all(np.array_equal(x, y) for x, y in zip(a, b)), "ok": int((a[3] == 0).sum())}
    m.close()
txt = json.dumps(report, indent=1)
print(txt)
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write(txt + "\n")
