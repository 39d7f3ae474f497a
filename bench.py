#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on BASELINE.json's configs, one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg4|cfg5|strong|k2]
                  [--dump-outputs DIR]
  (N > 1: launched by torchrun, one rank per GPU; RANK / LOCAL_RANK / WORLD_SIZE from the env)

--dump-outputs DIR (cfg2 / strong): after the timed steps, rank 0 writes what its last timed CorrelateScan returned for
its batch as DIR/{response,pose,covariance,status,tie_count}.npy (float64; status and tie counts are integers held
exactly).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.

--workload cfg2 (default, the headline; config.workload = "cfg2"): B = 1024 synthetic 1081-beam scans per GPU (Hokuyo
UTM-30LX model), each matched against its own 0.05 m correlation grid (one base scan, 20.05 m x 20.05 m ROI) with a direct
ScanMatcher::CorrelateScan over a 31 x 31 x 181 window (+-0.75 m @0.05 m, +-22.5 deg @0.25 deg), doPenalize=true
(SURVEY.md §8(d) cfg 2).  A "step" is one pass of the hot path over that batch.

  value : scan-matches/s with scans + grids already resident in HBM; timed region = K x b2s_matcher_correlate_scan
          (lookup lists + response sweep + best/tie-average/covariance + result D2H), CUDA events on the launching
          stream, barrier + synchronize on both sides, max over ranks.
  e2e   : the same metric through the host-buffer C-ABI calls a reference node would make
          (set_scans + add_scans (rasterise base scans) + correlate_scan) from PINNED host buffers, H2D + D2H inside
          the timed region.
  roofline : algorithmic bytes A1 = nX*nY*nA*N = 188 030 221 B per match (SURVEY.md §8(d)) x matches per launch
          / average k_sweep_window duration (CUDA events inside the library, same stream), against the measured HBM
          copy bandwidth in MEASURED_PEAKS.json.  K1 is an on-chip-gather kernel: the bytes are served from shared
          memory, so this is an EFFECTIVE bandwidth; `smem_gather` reports the same work against the
          shared-memory bank ceiling, which is the resource that actually binds.
  roofline_k2 : the metric's other half ("+ grid cells/s"): per K2 flavour A2 = 2 x cell bytes x V (V = Bresenham cell
          visits, SURVEY.md §8(d)) / kernel time vs the same HBM peak, DRAM traffic from the committed ncu captures.
  cpu_baseline : the reference's own single-threaded CorrelateScan (oracle/_ref, unmodified open_karto, -O2 -DNDEBUG)
          on a bounded sample of the same workload, rank 0 / N = 1 only.

Other workloads (each one JSON line with the same keys; all run under torchrun at 1/2/4/8 GPUs):
  cfg4   BASELINE cfg 4: windows 11x11x61 -> 61x61x361 on a 0.025 m grid, batch-sharded over the ranks
  cfg5   BASELINE cfg 5: loop-closure candidate chains of a many-lap trajectory enumerated by b2s_mapper (outdoor yaml),
         their coarse MatchScan batch-sharded over the ranks, then the CPU pose-graph solve
  strong a FIXED 1024 cfg-2 matches split over the ranks (strong scaling)
  k2     the K2 / front-end sections alone (grid cells/s)
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "creating-2d-laser-slam-from-scratch_b200"
D = 0.01745329251994329577
NX = NY = 31
NA = 181
NBEAMS = 1081
A1_BYTES = NX * NY * NA * NBEAMS  # 188 030 221 algorithmic bytes per scan-match
KERNELS_PER_STEP = 5  # k_bases, k_offsets_sorted, k_sweep_window (+ fused tail), k_sweep_generic (fall-through), k_reduce
METRIC = "scan-matches/s (1081-beam, 31x31x181 window)"
DTYPE = "u8 gather + i32 sum, f64 pose"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4", "cfg5", "strong", "k2"])
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--cpu-sample", type=int, default=48, help="matches timed for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-k2", action="store_true", help="skip the secondary grid-cells/s measurements")
    ap.add_argument("--quick", action="store_true", help="smaller secondary sections (development)")
    ap.add_argument("--nodes", type=int, default=5000, help="cfg5: key frames of the trajectory")
    ap.add_argument("--min-seconds", type=float, default=0.0, help="repeat the timed steps until at least this long")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("cfg2", "strong")):
        ap.error("--dump-outputs covers the cfg2 / strong CorrelateScan path of --impl ours")
    return args


def dump_outputs(directory, out):
    """The arrays correlate_scan returned (response, pose, covariance, status, tie_count) as float64 .npy files."""
    os.makedirs(directory, exist_ok=True)
    for name, a in zip(("response", "pose", "covariance", "status", "tie_count"), out):
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


def cfg2_config(B, world):
    return {"workload": "cfg2", "batch_per_gpu": B, "beams": NBEAMS, "window": [NX, NY, NA], "grid_res_m": 0.05,
            "grid_bytes": 165240, "base_scans": 1, "parallelism": f"batch-shard x{world}",
            "l2_policy": f"inputs larger than L2 ({B} grids x 165 KB = {B * 165240 / 1e6:.0f} MB resident, "
                         f"{B * NA * NX * NY * 4 / 1e6:.0f} MB volume per step)"}


def make_workload(synth, batch, rank, base=1_000_000):
    cases = [synth.make_match_case(base + rank * batch + i) for i in range(batch)]
    ranges = np.stack([c.ranges for c in cases])
    poses = np.stack([c.odom_pose for c in cases])
    bran = np.stack([c.base_ranges for c in cases])[:, None, :]
    bpos = np.stack([c.base_pose for c in cases])[:, None, :]
    return ranges, poses, bran, bpos


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag, self.proc = gpu_index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def host_desc():
    try:
        model = [l.split(":")[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        model = "unknown"
    return f"{model} x{os.cpu_count()}"


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(name, batch=None):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` summaries (profiles/dram_traffic.json)."""
    path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if not os.path.exists(path):
        return None, None
    t = json.load(open(path)).get(name)
    if not t or (batch is not None and int(t.get("batch", batch)) != batch):
        return None, None
    return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"]), t.get("source")


# ------------------------------------------------------------------------------------------------ CPU reference legs

def cpu_baseline(pkg, n_sample, ranges, poses, bran, bpos):
    """The reference's own single-threaded CorrelateScan on the first n_sample matches of the workload."""
    from oracle import ref
    synth = pkg.synth
    A, R = 22.5 * D, 0.25 * D
    if ref.available(ndebug=True):
        kind, secs = "reference", []
        s = ref.RefSession(ref.default_matcher_params(1.5, 0.05, 0.03, 9.25), synth.Laser(), ndebug=True)
        for i in range(n_sample):
            b = s.add_scan(bran[i, 0], bpos[i, 0])
            c = s.add_scan(ranges[i], poses[i])
            s.set_grid_from_scans(c, [b])
            secs.append(float(s.time_correlate(c, s.sensor_pose(c), (0.75, 0.75), (0.05, 0.05), A, R, True, False, 1)[0]))
        s.close()
    else:
        from oracle import port
        kind, secs = "port", []
        abi = pkg.abi
        for i in range(n_sample):
            pm = port.PortMatcher(abi.matcher_params(1.5, 0.05, 0.03, 9.25), abi.laser_from(synth.Laser()))
            pm.set_scan(ranges[i], poses[i])
            pm.add_scans(bran[i], bpos[i])
            t = time.perf_counter()
            pm.correlate_scan(pm.sp, abi.Search(0.75, 0.75, 0.05, 0.05, A, R, 1, 0))
            secs.append(time.perf_counter() - t)
    secs = np.array(secs)
    return {"value": float(1.0 / np.median(secs)), "unit": "scan-matches/s", "cores": 1, "kind": kind,
            "sample": f"{n_sample} of the {len(ranges)} cfg2 matches, ScanMatcher::CorrelateScan 31x31x181, "
                      f"median {np.median(secs) * 1e3:.1f} ms/match, g++ -O2 -DNDEBUG, 1 thread",
            "host": host_desc()}


_REF_STATE = {}


def _ref_init(n_cases, seed0):
    """Pool initialiser: one persistent reference ScanMatcher session per worker process with its matches preloaded
    (the reference is single-threaded and not re-entrant: one session per process)."""
    sys.path.insert(0, ROOT)
    pkg = importlib.import_module(PKG)
    from oracle import port, ref
    import multiprocessing as mp
    ident = mp.current_process()._identity
    wid = ident[0] if ident else 0
    cases = [pkg.synth.make_match_case(seed0 + 1000 * wid + i) for i in range(n_cases)]
    st = {"pkg": pkg, "cases": cases, "kind": "port"}
    if ref.available(ndebug=True):
        s = ref.RefSession(ref.default_matcher_params(1.5, 0.05, 0.03, 9.25), pkg.synth.Laser(), ndebug=True)
        st["session"] = s
        st["ids"] = [(s.add_scan(c.base_ranges, c.base_pose), s.add_scan(c.ranges, c.odom_pose)) for c in cases]
        st["kind"] = "reference"
    _REF_STATE.update(st)


def _ref_step(n_matches):
    """One worker's share of a step: n_matches full matches (grid build + CorrelateScan) on its own session."""
    st = _REF_STATE
    A, R = 22.5 * D, 0.25 * D
    t0 = time.perf_counter()
    if st["kind"] == "reference":
        s = st["session"]
        for k in range(n_matches):
            b, c = st["ids"][k % len(st["ids"])]
            s.set_grid_from_scans(c, [b])
            s.correlate_scan(c, s.sensor_pose(c), (0.75, 0.75), (0.05, 0.05), A, R, True, False)
    else:
        from oracle import port
        pkg = st["pkg"]
        abi = pkg.abi
        for k in range(n_matches):
            c = st["cases"][k % len(st["cases"])]
            pm = port.PortMatcher(abi.matcher_params(1.5, 0.05, 0.03, 9.25), abi.laser_from(pkg.synth.Laser()))
            pm.set_scan(c.ranges, c.odom_pose)
            pm.add_scans(c.base_ranges, c.base_pose)
            pm.correlate_scan(pm.sp, abi.Search(0.75, 0.75, 0.05, 0.05, A, R, 1, 0))
    return n_matches, time.perf_counter() - t0, st["kind"]


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores (one persistent
    single-threaded ScanMatcher session per worker process), same metric / config keys; each step is a bounded sample
    of the workload: 8 matches per worker."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = max(1, min(os.cpu_count() or 1, 64))
    per_worker = 8
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores, initializer=_ref_init, initargs=(per_worker, 2_000_000)) as pool:
        def step():
            t0 = time.perf_counter()
            out = pool.map(_ref_step, [per_worker] * cores, chunksize=1)
            return sum(o[0] for o in out), time.perf_counter() - t0, out[0][2], [o[1] for o in out]
        for _ in range(max(args.warmup, 1)):
            step()
        t_total, n_total, kind, busy = 0.0, 0, "reference", []
        for _ in range(args.steps):
            n, t, kind, b = step()
            n_total += n
            t_total += t
            busy += b
    value = n_total / t_total
    per_core = per_worker / float(np.median(busy))
    line = {"impl": "reference", "metric": METRIC, "value": value,
            "unit": "scan-matches/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_total / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": cfg2_config(args.batch, world),
            "cpu_baseline": {"value": value, "unit": "scan-matches/s", "cores": cores, "kind": kind,
                             "per_core": per_core,
                             "sample": f"{cores * per_worker} matches per step ({per_worker} per worker process, persistent "
                                       f"sessions, incl. the grid build of every match), {args.steps} steps; the full "
                                       f"cfg2 batch is {args.batch} matches per GPU",
                             "host": host_desc()},
            "e2e": {"value": value, "unit": "scan-matches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------ shared plumbing

class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (VERSION prints a banner there)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.pkg = importlib.import_module(PKG)
        self.stream = torch.cuda.Stream(device=self.local)  # a real (non-default) stream shared with the library, so that
        torch.cuda.set_stream(self.stream)                  # torch.cuda.Event brackets exactly the library's launches

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, ms):
        t = self.torch.tensor([ms], device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, v):
        t = self.torch.tensor([v], device="cuda", dtype=self.torch.float64)
        if self.world == 1:
            return [float(v)]
        outs = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(outs, t)
        return [float(o.item()) for o in outs]

    def timed(self, fn, steps, min_seconds=0.0):
        """barrier + synchronize, K x fn() between two CUDA events on the library's stream, barrier + synchronize;
        returns (max-over-ranks ms, per-rank ms list, steps actually run).  min_seconds repeats the K steps."""
        torch = self.torch
        total_ms, done, per_rank = 0.0, 0, None
        while True:
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            for _ in range(steps):
                fn()
            e1.record(self.stream)
            self.barrier()
            ms = e0.elapsed_time(e1)
            ranks = self.gather(ms)
            per_rank = ranks if per_rank is None else [a + b for a, b in zip(per_rank, ranks)]
            total_ms += max(ranks)
            done += steps
            if total_ms * 1e-3 >= min_seconds:
                break
        return total_ms, per_rank, done

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def oracle_check_matches(pkg, params, laser, ranges, poses, bran, bpos, search, got, idx):
    """multi_gpu_exact-style self check: matches `idx` of this rank's batch against the CPU restatement."""
    from oracle import port
    worst, ok = 0.0, True
    for b in idx:
        pm = port.PortMatcher(params, laser)
        pm.set_scan(ranges[b], poses[b])
        pm.add_scans(bran[b], bpos[b])
        rc, res = pm.correlate_scan(pm.sp, search)
        if rc != 0 or got[3][b] != 0:
            ok = ok and (rc == got[3][b])
            continue
        d = max(abs(got[0][b] - res.response), float(np.abs(got[1][b] - np.array(res.pose[:])).max()))
        worst = max(worst, d)
        ok = ok and d <= 1e-9
    return {"checked": len(idx), "ok": bool(ok), "max_abs_diff": worst, "vs": "oracle C restatement (pinned to the reference)"}


# ------------------------------------------------------------------------------------------------ K2 + front ends

def bench_k2(pkg, local, quick=False):
    """Secondary metric of BASELINE.json ("+ grid cells/s"): K2c Karto full-map rebuild, K2a Hector update (single
    stream, one-call stream, B independent maps), K2b GMapping, and the front ends built on K1/K2/K3.
    cells/s = Bresenham cell visits per second (library-reported V, SURVEY.md §8(d)); achieved = A2 x rate with
    A2 = 2 x cell bytes x V (4 B Karto counter, 8 B Hector cell, 16 B GMapping cell).
    Returns (sections, roofline_k2)."""
    import torch
    abi, synth = pkg.abi, pkg.synth
    O, H = pkg.load("occgrid"), pkg.load("hector")
    laser = synth.Laser()
    peak, peak_src = hbm_peak()
    out, roof = {}, {"peak": peak, "peak_source": peak_src, "unit": "GB/s", "bound": "hbm",
                     "note": "A2 = 2 x cell bytes x V; single resident maps sit in L2 (atomic-throughput bound), the "
                             "batched Hector case streams B maps larger than L2 through HBM"}

    def roof_row(name, a2_bytes, seconds, kernel, traffic_key=None, batch=None, launches=None):
        ach = a2_bytes / seconds / 1e9
        tr, src = committed_traffic(traffic_key or kernel, batch)
        roof[name] = {"kernel": kernel, "achieved": ach, "frac": ach / peak, "algorithmic_bytes": a2_bytes,
                      "seconds": seconds, "traffic": tr, "traffic_source": src}
        if tr and launches:  # DRAM bytes per launch (ncu) x launches in the timed region / time: the physical HBM fraction
            roof[name]["dram_GBps_from_traffic"] = tr * launches / seconds / 1e9
            roof[name]["dram_frac_from_traffic"] = tr * launches / seconds / 1e9 / peak

    # --- K2c: OccupancyGrid::CreateFromScans over a 2000-scan trajectory (what SlamKarto::updateMap rebuilds)
    n_scans = 400 if quick else 2000
    world, poses, ranges = synth.make_trajectory(21, min(n_scans, 200), laser, step_xy=0.25, step_th_deg=6)
    reps = n_scans // len(poses)
    poses, ranges = np.tile(poses, (reps, 1)), np.tile(ranges, (reps, 1))
    al = abi.laser_from(laser)
    for _ in range(2):
        g = O.OccupancyGrid(al, ranges, poses, 0.05, device=local)
        g.close()
    t_ray, t_wall, visits = [], [], 0
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g = O.OccupancyGrid(al, ranges, poses, 0.05, device=local)
        torch.cuda.synchronize()
        t_wall.append(time.perf_counter() - t0)
        t_ray.append(g.last_timing()["raytrace_ms"] * 1e-3)
        visits = int(g.info.cell_visits)
        dims = (g.info.width, g.info.height)
        g.close()
    ray, wall = float(np.median(t_ray)), float(np.median(t_wall))
    out["karto_occupancy_grid"] = {
        "scans": n_scans, "beams": 1081, "map_cells": list(dims), "cell_visits": visits,
        "cells_per_s_kernel": visits / ray, "cells_per_s_e2e": visits / wall, "scans_per_s_e2e": n_scans / wall,
        "raytrace_ms": ray * 1e3, "e2e_ms": wall * 1e3,
        "achieved_GBps": 2 * 4 * visits / ray / 1e9}
    roof_row("karto_occupancy_grid", 2 * 4 * visits, ray, "k_raytrace", batch=n_scans, launches=1)
    try:  # the reference's own OccupancyGrid::CreateFromScans on a 70-scan sample (survey probe shape), 1 thread
        from oracle import ref
        if ref.available(ndebug=True):
            rs = ref.RefSession(ref.default_matcher_params(1.5, 0.05, 0.03, 9.25), laser, ndebug=True)
            ids = [rs.add_scan(ranges[i], poses[i]) for i in range(70)]
            secs = rs.time_occgrid(ids, 0.05, reps=5)
            rs.close()
            out["karto_occupancy_grid"]["cpu_reference"] = {
                "scans_per_s": 70 / float(np.median(secs)), "sample": "70 scans x 1081 beams, 1 thread, -O2 -DNDEBUG",
                "ms": float(np.median(secs)) * 1e3}
    except Exception as e:
        out["karto_occupancy_grid"]["cpu_reference"] = {"error": repr(e)}

    # --- K2a + K3: Hector stream (cfg 3 shape): HectorSlamProcessor::update per scan = 3-level GN match + gated
    #     3-level log-odds update on a 1000^2 @0.05 m map (50 m x 50 m), node defaults (0.4/0.9 factors, 0.4 m / 0.9 rad gate)
    n_stream = 300 if quick else 10000  # cfg 3: a 10 000-scan stream
    world, poses, ranges = synth.make_trajectory(22, n_stream, laser, step_xy=0.05, step_th_deg=1.0)
    pts = [H.scan_to_data_container(ranges[i], laser, 0.05, max_dist=30.0, min_dist=0.2) for i in range(n_stream)]
    kw = dict(resolution=0.05, size_x=1000, size_y=1000, start=(0.5, 0.5), levels=3, update_free=0.4, update_occupied=0.9,
              min_dist=0.4, min_angle=0.9)
    hstream = {"scans": n_stream, "levels": 3,
               "note": "the node's loop (hint = last scan-match pose).  per_scan = one b2s_hector_slam_update call per LaserScan "
                       "(one cooperative launch: match + gate + update on the device, pose back through a host-mapped mailbox); "
                       "stream = the whole recording in one b2s_hector_slam_process_stream call (no host round trip between "
                       "scans).  exact = bit-identical to the reference (sequential float32 sums: 14 x 1081 dependent adds per "
                       "scan); fast = tree sums, poses within 1e-4"}
    stream_poses_by_mode = {}
    for exact in (True, False):
        tag = "exact" if exact else "fast"
        hs = H.HectorSlam(device=local, exact=exact, **kw)
        est = poses[0].astype(np.float32)
        n_ps = min(n_stream, 2000)
        est, _ = hs.update(pts[0], (0, 0), est)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(1, n_ps):
            est, cov = hs.update(pts[i], (0, 0), est)
        st = hs.stats()
        dt = time.perf_counter() - t0
        hstream[f"per_scan_{tag}"] = {"scans": n_ps - 1, "scans_per_s": (n_ps - 1) / dt, "us_per_scan": 1e6 * dt / (n_ps - 1),
                                      "map_updates": st["updated"], "last_match_ms": st["match_ms"],
                                      "last_update_ms": st["update_ms"],
                                      "final_xy_err_m": float(np.abs(est[:2] - poses[n_ps - 1][:2]).max())}
        hs.close()
        hs = H.HectorSlam(device=local, exact=exact, **kw)
        hs.process_stream(pts[:16], (0, 0), first_hint=poses[0].astype(np.float32))  # warm-up (allocations, module load)
        hs.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p_all, u_all, _ = hs.process_stream(pts, (0, 0), first_hint=poses[0].astype(np.float32))
        dt = time.perf_counter() - t0
        st = hs.stats()
        stream_poses_by_mode[tag] = p_all
        hstream[f"stream_{tag}"] = {"scans": n_stream, "scans_per_s": n_stream / dt, "us_per_scan": 1e6 * dt / n_stream,
                                    "map_updates": int(u_all.sum()), "cell_visits": st["cell_visits"],
                                    "cells_per_s": st["cell_visits"] / dt,
                                    "final_xy_err_m": float(np.abs(p_all[-1][:2] - poses[-1][:2]).max()),
                                    "h2d_bytes": int(sum(len(p) for p in pts) * 8), "d2h_bytes": n_stream * 64}
        hs.close()
    hstream["scans_per_s"] = hstream["stream_exact"]["scans_per_s"]
    dpose = np.abs(stream_poses_by_mode["fast"] - stream_poses_by_mode["exact"])
    dpose[:, 2] = np.abs((dpose[:, 2] + np.pi) % (2 * np.pi) - np.pi)
    hstream["fast_vs_exact_max_abs_pose_diff"] = {"xy_m": float(dpose[:, :2].max()), "theta_rad": float(dpose[:, 2].max()),
                                                  "note": "self-driven streams (each mode feeds its own poses back as hints)"}
    out["hector_stream"] = hstream
    stream_ranges, stream_poses = ranges, poses  # reused by the PL-ICP odometry stream below
    # every-scan mapping (gate off): the K2a update rate of ONE map (L2-resident)
    hs = H.HectorSlam(device=local, **dict(kw, min_dist=0.0, min_angle=0.0))
    n_map = min(n_stream, 1000)
    hs.process_stream(pts[:4], (0, 0), pose_hints=poses[:4].astype(np.float32), map_without_matching=True)
    hs.reset()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    hs.process_stream(pts[:n_map], (0, 0), pose_hints=poses[:n_map].astype(np.float32), map_without_matching=True)
    dt = time.perf_counter() - t0
    st = hs.stats()
    out["hector_mapping_only"] = {"scans": n_map, "scans_per_s": n_map / dt, "cell_visits": st["cell_visits"],
                                  "cells_per_s": st["cell_visits"] / dt,
                                  "achieved_GBps": 2 * 8 * st["cell_visits"] / dt / 1e9,
                                  "note": "updateByScan with given poses (map_without_matching), one map, one-call stream; "
                                          "level 0 only receives data"}
    roof_row("hector_single_map", 2 * 8 * st["cell_visits"], dt, "k_hs_stream (update passes)")
    hs.close()
    # B independent maps (SURVEY.md §8(e): Hector shards over independent maps): B x 1000^2 x 3-level maps = B x 26 MB
    # of cell state, larger than L2 -> the update streams through HBM.  Scans resident on the device.
    try:
        Bm = 16 if quick else 128
        steps = 8 if quick else 24
        cap = max(len(p) for p in pts)
        hb = H.HectorSlam(device=local, batch=Bm, max_points=cap, **dict(kw, min_dist=0.0, min_angle=0.0))
        hp = np.zeros((steps, Bm, cap, 2), np.float32)
        hn = np.zeros((steps, Bm), np.int32)
        hh = np.zeros((steps, Bm, 3), np.float32)
        for s_ in range(steps):
            for b in range(Bm):
                i = (s_ * 7 + b * 13) % n_stream
                hp[s_, b, :len(pts[i])] = pts[i]
                hn[s_, b] = len(pts[i])
                hh[s_, b] = poses[i]
        dp, dn, dh = torch.from_numpy(hp).cuda(), torch.from_numpy(hn).cuda(), torch.from_numpy(hh).cuda()
        torch.cuda.synchronize()
        for s_ in range(3):
            hb.update_batch_device(dp[s_].data_ptr(), dn[s_].data_ptr(), cap, (0, 0), dh[s_].data_ptr(), True)
        hb.sync()
        v0 = hb.stats()["cell_visits"]
        t0 = time.perf_counter()
        for s_ in range(3, steps):
            hb.update_batch_device(dp[s_].data_ptr(), dn[s_].data_ptr(), cap, (0, 0), dh[s_].data_ptr(), True)
        hb.sync()
        dt = time.perf_counter() - t0
        v = hb.stats()["cell_visits"] - v0
        out["hector_batched_maps"] = {"maps": Bm, "steps": steps - 3, "scans_per_s": Bm * (steps - 3) / dt, "cell_visits": v,
                                      "cells_per_s": v / dt, "ms_per_step": 1e3 * dt / (steps - 3),
                                      "map_state_MB": Bm * 1000 * 1000 * 32 * (1 + 0.25 + 0.0625) / 1e6,
                                      "note": "mapping only, given poses; scans already in HBM (b2s_hector_slam_update_batch_device)"}
        roof_row("hector_batched_maps", 2 * 8 * v, dt, "k_hs_mark + k_hs_apply", traffic_key="k_hs_batched_update", batch=Bm, launches=steps - 3)
        hb.close()
        # the same B maps fed from a 44 m x 44 m hall (rays up to 30 m): every update sweeps most of the 1000^2 map, so the
        # cell state (B x 26 MB) streams through HBM instead of sitting in L2
        _, hp2, hr2 = synth.make_trajectory(29, 48, laser, half_w=22.0, half_h=22.0, step_xy=0.3, step_th_deg=8, n_boxes=24)
        pts2 = [H.scan_to_data_container(hr2[i], laser, 0.05, max_dist=30.0, min_dist=0.2) for i in range(len(hp2))]
        cap2 = max(len(p) for p in pts2)
        hb = H.HectorSlam(device=local, batch=Bm, max_points=cap2, **dict(kw, min_dist=0.0, min_angle=0.0))
        hq = np.zeros((steps, Bm, cap2, 2), np.float32); hm = np.zeros((steps, Bm), np.int32); hg = np.zeros((steps, Bm, 3), np.float32)
        for s_ in range(steps):
            for b in range(Bm):
                i = (s_ * 5 + b * 11) % len(pts2)
                hq[s_, b, :len(pts2[i])] = pts2[i]; hm[s_, b] = len(pts2[i]); hg[s_, b] = hp2[i]
        dq, dm, dg = torch.from_numpy(hq).cuda(), torch.from_numpy(hm).cuda(), torch.from_numpy(hg).cuda()
        torch.cuda.synchronize()
        for s_ in range(3):
            hb.update_batch_device(dq[s_].data_ptr(), dm[s_].data_ptr(), cap2, (0, 0), dg[s_].data_ptr(), True)
        hb.sync()
        v0 = hb.stats()["cell_visits"]
        t0 = time.perf_counter()
        for s_ in range(3, steps):
            hb.update_batch_device(dq[s_].data_ptr(), dm[s_].data_ptr(), cap2, (0, 0), dg[s_].data_ptr(), True)
        hb.sync()
        dt = time.perf_counter() - t0
        v = hb.stats()["cell_visits"] - v0
        out["hector_batched_maps_hall"] = {"maps": Bm, "steps": steps - 3, "scans_per_s": Bm * (steps - 3) / dt, "cell_visits": v,
                                           "cells_per_s": v / dt, "ms_per_step": 1e3 * dt / (steps - 3),
                                           "note": "44 m x 44 m hall, 30 m rays: the swept region of every map is ~800 x 800 cells"}
        roof_row("hector_batched_maps_hall", 2 * 8 * v, dt, "k_hs_mark + k_hs_apply", traffic_key="k_hs_batched_update_hall", batch=Bm, launches=steps - 3)
        # the same handle as B SLAM processors (match + gate + update per step)
        hb.close()
        hb = H.HectorSlam(device=local, batch=Bm, max_points=cap, **kw)
        for s_ in range(3):
            hb.update_batch_device(dp[s_].data_ptr(), dn[s_].data_ptr(), cap, (0, 0), dh[s_].data_ptr(), False)
        hb.sync()
        t0 = time.perf_counter()
        for s_ in range(3, steps):
            hb.update_batch_device(dp[s_].data_ptr(), dn[s_].data_ptr(), cap, (0, 0), dh[s_].data_ptr(), False)
        hb.sync()
        dt = time.perf_counter() - t0
        out["hector_batched_slam"] = {"processors": Bm, "steps": steps - 3, "scans_per_s": Bm * (steps - 3) / dt,
                                      "ms_per_step": 1e3 * dt / (steps - 3), "mode": "exact",
                                      "note": "B independent HectorSlamProcessors, one scan each per step (3-level match + gated update)"}
        hb.close()
    except Exception as e:
        out["hector_batched_maps"] = {"error": repr(e)}
    try:  # the reference's own HectorSlamProcessor (unmodified headers + Eigen stand-in), 1 thread, same stream sample
        from oracle import ref_hector as rh
        if rh.available():
            n_ref = min(n_stream, 300)
            rp = rh.RefHectorProcessor(**kw)
            e = poses[0].astype(np.float32)
            t0 = time.perf_counter()
            for i in range(n_ref):
                e, _ = rp.update(pts[i], (0, 0), e)
            dt = time.perf_counter() - t0
            rp.close()
            out["hector_stream"]["cpu_reference"] = {"scans_per_s": n_ref / dt, "sample": f"first {n_ref} scans of the same stream, "
                                                     "HectorSlamProcessor::update, g++ -O2, 1 thread"}
            rp = rh.RefHectorProcessor(**dict(kw, min_dist=0.0, min_angle=0.0))
            t0 = time.perf_counter()
            for i in range(n_ref):
                rp.update(pts[i], (0, 0), poses[i].astype(np.float32), True)
            dt = time.perf_counter() - t0
            rp.close()
            out["hector_mapping_only"]["cpu_reference"] = {"scans_per_s": n_ref / dt, "sample": f"{n_ref} scans, updateByScan with "
                                                           "given poses, g++ -O2, 1 thread"}
    except Exception as e:
        out["hector_stream"]["cpu_reference"] = {"error": repr(e)}

    # --- K2b: GMapping ComputeMap (gmapping.cc:127-242): one full counter map per scan, 2000 x 2000 cells @0.05 m
    try:
        GM = pkg.load("gmapping")
        from oracle import port as _port
        ang = (np.float32(laser.min_angle) + np.arange(1081, dtype=np.float32) * np.float32(laser.angular_resolution)).astype(np.float64)
        n_g = 50 if quick else 400
        gr = [ranges[i].astype(np.float32).astype(np.float64) for i in range(n_g)]
        gm = GM.GMap(-50, -50, 50, 50, 0.05, device=local)
        gm.compute_map(gr[0], ang, (0.0, 0.0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(1, n_g):
            gm.compute_map(gr[i], ang, (float(poses[i, 0]), float(poses[i, 1])))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        vg = int(gm.cells()[1].sum())
        out["gmapping_compute_map"] = {"scans": n_g - 1, "scans_per_s": (n_g - 1) / dt, "cell_visits": vg, "cells_per_s": vg / dt,
                                       "achieved_GBps": 2 * 16 * vg / dt / 1e9, "map_cells": [gm.size_x, gm.size_y],
                                       "note": "host ranges in, counters stay on the device (one call per scan)"}
        roof_row("gmapping_compute_map", 2 * 16 * vg, dt, "k_gm_update")
        gm.close()
        pg = _port.PortGMap(-50, -50, 50, 50, 0.05)
        n_c = min(n_g, 40)
        t0 = time.perf_counter()
        for i in range(n_c):
            pg.compute_map(gr[i], ang, (float(poses[i, 0]), float(poses[i, 1])))
        dt = time.perf_counter() - t0
        out["gmapping_compute_map"]["cpu_reference"] = {"scans_per_s": n_c / dt, "kind": "port (oracle/gmapping_oracle.c, pinned to "
                                                        "the reference's grid headers)", "sample": f"{n_c} scans, 1 thread, -O2"}
    except Exception as e:
        out["gmapping_compute_map"] = {"error": repr(e)}

    # --- K1 beyond the headline shape: the default two-stage MatchScan (coarse stride-2 + fine)
    M = pkg.load("matcher")
    try:
        Bm = 256 if quick else 1024
        cases = [synth.make_match_case(3_000_000 + i) for i in range(Bm)]
        mr, mp = np.stack([c.ranges for c in cases]), np.stack([c.odom_pose for c in cases])
        mbr, mbp = np.stack([c.base_ranges for c in cases])[:, None, :], np.stack([c.base_pose for c in cases])[:, None, :]
        mm = M.ScanMatcher(abi.matcher_params(1.5, 0.05, 0.03, 9.25), al, max_batch=Bm, max_base_scans=1, device=local)
        mm.match_scan_host(mr, mp, mbr, mbp)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            r_ms = mm.match_scan_host(mr, mp, mbr, mbp)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 3
        truth = np.stack([c.true_pose for c in cases])
        out["match_scan_two_stage"] = {"batch": Bm, "shape": "coarse 16x16x21 (stride 2) + fine 3x3x11, 1.5 m / 0.05 m, 1 base scan",
                                       "matches_per_s_e2e": Bm / dt, "ms": dt * 1e3,
                                       "median_xy_err_m": float(np.median(np.abs(r_ms[1][:, :2] - truth[:, :2]).max(axis=1)))}
        mm.close()
    except Exception as e:
        out["k1_extras_error"] = repr(e)
    # --- lesson6 front end (SURVEY.md §8(f).1): karto::Mapper::Process per key frame through b2s_mapper_process with the
    #     shipped indoor yaml (lesson6/config/mapper_params.yaml: 0.3 m / 0.01 m sequential window on a 2431^2 grid,
    #     110-scan running buffer, 10 m / 0.05 m loop window, response expansion on); near chains / loop candidates batched.
    #     Two streams: laps of a 2 m circle in the small room (no loop candidates: every scan stays near-linked), and two
    #     laps of a 9 m circle in a 28 m x 24 m hall, where the second lap meets the first as loop-closure candidates.
    try:
        MPm = pkg.load("mapper")
        lm = synth.Laser(range_threshold=12.0)
        yaml = dict(scan_buffer_size=110, scan_buffer_maximum_scan_distance=100.0, link_match_minimum_response_fine=0.1,
                    link_scan_maximum_distance=1.5, loop_search_maximum_distance=10.0, loop_match_minimum_chain_size=5,
                    loop_match_maximum_variance_coarse=9.0, loop_match_minimum_response_coarse=0.35,
                    loop_match_minimum_response_fine=0.45, minimum_travel_heading=0.174, loop_search_size=10.0,
                    both_distance_variance_penalty=0.25, both_angle_variance_penalty=0.01,
                    both_fine_search_angle_offset=0.00349, both_coarse_search_angle_offset=0.349,
                    both_coarse_angle_resolution=0.0349, both_use_response_expansion=1)
        prm = MPm.default_params(12.0, **yaml)
        from oracle import ref as _ref
        for key, n_map, traj, n_ref in (
                ("karto_mapper_stream", 120 if quick else 400, dict(radius=2.0, step=0.25), 150),
                ("karto_mapper_stream_loops", 120 if quick else 520,
                 dict(radius=2.0, step=0.25) if quick else dict(radius=9.0, step=0.25, half_w=14.0, half_h=12.0, n_boxes=12), 520)):
            _, tru, odo, rng_m = synth.make_loop_trajectory(17, n_map, lm, **traj)
            mp_ = MPm.Mapper(prm, abi.laser_from(lm), device=local)
            n_warm = 30  # the first frames create the matcher handles (device + pinned allocations, ~0.2-1.5 s once per mapper)
            for i in range(n_warm):
                mp_.process(rng_m[i], odo[i], 0.1 * i)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(n_warm, n_map):
                mp_.process(rng_m[i], odo[i], 0.1 * i)
            dt = time.perf_counter() - t0
            stm = mp_.stats()
            out[key] = {"key_frames": n_map - n_warm, "scans_per_s": (n_map - n_warm) / dt, "ms_per_scan": 1e3 * dt / (n_map - n_warm),
                        "untimed_first_frames": n_warm, "match_scan_calls": stm["match_calls"], "device_batches": stm["batches"],
                        "loop_candidates": stm["loop_candidates"], "loops_closed": stm["loops_closed"],
                        "edges": int(len(mp_.edges()[0])),
                        "max_xy_err_m": float(np.abs(mp_.poses()[:, :2] - tru[:, :2]).max()),
                        "config": "lesson6/config/mapper_params.yaml (no back end), 1081 beams, range threshold 12 m; " + repr(traj)}
            mp_.close()
            if _ref.available(ndebug=True):  # the reference Mapper on the SAME frames (the timed ones included)
                n_r = min(n_map, n_ref)
                rm = _ref.RefMapper(prm, lm, ndebug=True)
                for i in range(min(n_warm, n_r)):
                    rm.process(rng_m[i], odo[i], 0.1 * i)
                t0 = time.perf_counter()
                done = 0
                for i in range(n_warm, n_r):
                    rm.process(rng_m[i], odo[i], 0.1 * i)
                    done += 1
                    if time.perf_counter() - t0 > 90.0:
                        break
                dt = time.perf_counter() - t0
                rm.close()
                out[key]["cpu_reference"] = {"scans_per_s": done / dt, "key_frames": done,
                                             "sample": f"key frames {n_warm}..{n_warm + done} of the same stream, karto::Mapper::Process, "
                                                       "-O2 -DNDEBUG, 1 thread (capped at 90 s)"}
    except Exception as e:
        out["karto_mapper_stream"] = {"error": repr(e)}
    # --- K3 (lesson3): batched PL-ICP, 1024 independent scan pairs with odometry-like motion
    P = pkg.load("plicp")
    nb = 256 if quick else 1024
    rng = np.random.default_rng(5)
    theta = laser.min_angle + np.arange(laser.n_readings) * laser.angular_resolution
    world = synth.make_world(33)
    refs, sens, truth = [], [], []
    for i in range(64):
        pa = np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(-np.pi, np.pi)])
        d = np.array([rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1), rng.uniform(-0.05, 0.05)])
        c, s_ = np.cos(pa[2]), np.sin(pa[2])
        pb = np.array([pa[0] + c * d[0] - s_ * d[1], pa[1] + s_ * d[0] + c * d[1], pa[2] + d[2]])
        refs.append(synth.cast_scan(world, pa, laser, rng)); sens.append(synth.cast_scan(world, pb, laser, rng)); truth.append(d)
    reps = nb // 64
    refs, sens, truth = np.tile(np.stack(refs), (reps, 1)), np.tile(np.stack(sens), (reps, 1)), np.tile(np.stack(truth), (reps, 1))
    guess = np.zeros((nb, 3))
    ip = abi.icp_params()
    P.match(ip, refs, sens, theta, 0.1, 30.0, guess, device=local)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    x, valid, iters, nvalid, err = P.match(ip, refs, sens, theta, 0.1, 30.0, guess, device=local)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["plicp_batch"] = {"pairs": nb, "pairs_per_s_e2e": nb / dt, "ms": dt * 1e3, "valid": int(valid.sum()),
                          "mean_iterations": float(iters.mean()),
                          "median_xy_err_m": float(np.median(np.abs(x[:, :2] - truth[:, :2]).max(axis=1))),
                          "note": "sigma = 1 cm range noise; host buffers in, results out (H2D + kernel + D2H); parity unpinned"}
    try:  # CPU baseline of the same pairs: the restatement (CSM itself is absent: parity unpinned)
        from oracle import port as _port
        n_c = 24
        t0 = time.perf_counter()
        for i in range(n_c):
            _port.plicp_match(ip, refs[i], sens[i], theta, 0.1, 30.0, guess[i])
        dt = time.perf_counter() - t0
        out["plicp_batch"]["cpu_reference"] = {"pairs_per_s": n_c / dt, "kind": "port (oracle/plicp_oracle.c, restated from the paper; "
                                               "PARITY UNPINNED — CSM is not in the reference tree)", "sample": f"{n_c} pairs, 1 thread, -O2"}
    except Exception as e:
        out["plicp_batch"]["cpu_reference"] = {"error": repr(e)}
    # --- cfg 3's other half: the lesson3 PL-ICP odometry over the same 10 000-scan stream (plicp_odometry.cc:191-436): scan i
    #     against scan i-1 with a zero first guess; consecutive pairs are independent, so the stream is ONE batched call
    try:
        n_od = len(stream_ranges) - 1
        t0 = time.perf_counter()
        xo, vo, _, _, _ = P.match(ip, stream_ranges[:-1], stream_ranges[1:], theta, 0.1, 30.0, np.zeros((n_od, 3)), device=local)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        pose = stream_poses[0].copy()  # dead-reckon the increments
        for i in range(n_od):
            c, s_ = np.cos(pose[2]), np.sin(pose[2])
            pose = np.array([pose[0] + c * xo[i, 0] - s_ * xo[i, 1], pose[1] + s_ * xo[i, 0] + c * xo[i, 1], pose[2] + xo[i, 2]])
        out["plicp_odometry_stream"] = {"pairs": n_od, "pairs_per_s_e2e": n_od / dt, "ms": dt * 1e3, "valid": int(vo.sum()),
                                        "final_xy_drift_m": float(np.abs(pose[:2] - stream_poses[-1][:2]).max()),
                                        "note": "pure scan-to-scan odometry, no map: drift accumulates; parity unpinned"}
    except Exception as e:
        out["plicp_odometry_stream"] = {"error": repr(e)}
    # --- lesson5 pre-stage: motion de-skew of a batch of scans (LidarUndistortion::CorrectLaserScan, one thread per beam)
    try:
        DS = pkg.load("deskew")
        nb_d, nbeam = (256 if quick else 2048), 1081
        rg = np.random.default_rng(5)
        rr = rg.uniform(0.5, 25.0, (nb_d, nbeam)).astype(np.float32)
        t0s = 100.0 + 0.1 * np.arange(nb_d)
        infos, T, X, Y, Z = [], [], [], [], []
        for b in range(nb_d):
            stamps = t0s[b] - 0.05 + np.arange(45) * 0.005
            t_end = t0s[b] + 0.1 / nbeam * (nbeam - 1)
            last, t, x, y, z = DS.integrate_imu(stamps, np.tile([0.1, -0.05, 0.8], (45, 1)), t0s[b], t_end, capacity=64)
            inf = DS.DeskewScan()
            inf.time_start, inf.time_increment, inf.range_min, inf.range_max = t0s[b], 0.1 / nbeam, 0.1, 30.0
            inf.use_imu = inf.use_odom = 1
            inf.imu_last, inf.odom_start_time, inf.odom_end_time = last, t0s[b] - 0.01, t_end - 0.004
            inc = DS.odom_increment([0, 0, 0, 0, 0, 0.1], [0.08, 0.01, 0, 0, 0, 0.18])
            inf.odom_incre[0], inf.odom_incre[1], inf.odom_incre[2] = inc
            infos.append(inf); T.append(t); X.append(x); Y.append(y); Z.append(z)
        T, X, Y, Z = (np.stack(a) for a in (T, X, Y, Z))
        a_min, a_inc = -2.35619449, 4.71238898 / (nbeam - 1)
        DS.undistort(rr[:8], a_min, a_inc, infos[:8], T[:8], X[:8], Y[:8], Z[:8], device=local)
        t0 = time.perf_counter()
        cloud = DS.undistort(rr, a_min, a_inc, infos, T, X, Y, Z, device=local)
        dt = time.perf_counter() - t0
        out["lidar_undistortion_batch"] = {"scans": nb_d, "beams": nbeam, "scans_per_s_e2e": nb_d / dt, "ms": dt * 1e3,
                                           "points_per_s": nb_d * nbeam / dt,
                                           "note": "host buffers in (ranges, IMU tables), corrected clouds out (H2D + kernel + D2H); "
                                                   "parity unpinned (PCL / Eigen are not in the reference tree)"}
        from oracle import port as _port
        n_c = 64
        t0 = time.perf_counter()
        ok = True
        for i in range(n_c):
            ref_cloud = _port.deskew_scan(rr[i], a_min, a_inc, infos[i], T[i], X[i], Y[i], Z[i])
            ok = ok and np.array_equal(ref_cloud.view(np.int32), cloud[i].view(np.int32))
        dt = time.perf_counter() - t0
        out["lidar_undistortion_batch"]["cpu_reference"] = {"scans_per_s": n_c / dt, "identical_to_device": bool(ok),
                                                            "kind": "port (oracle/deskew_oracle.c; PARITY UNPINNED)",
                                                            "sample": f"{n_c} scans, 1 thread, -O2 (ctypes call per scan)"}
    except Exception as e:
        out["lidar_undistortion_batch"] = {"error": repr(e)}
    return out, roof


def pose_graph_solve(pkg, nn, quick=False):
    """cfg 5's back end: the CPU pose-graph solve that follows the batched loop-closure matches (the library's own
    optimiser; the reference uses sba / SuiteSparse) on a synthetic nn-node, 4-lap graph."""
    MPg = pkg.load("mapper")
    per_lap = nn // 4
    th = np.arange(nn) * 2 * np.pi / per_lap
    tru = np.stack([20 * np.cos(th), 20 * np.sin(th), (th + np.pi / 2 + np.pi) % (2 * np.pi) - np.pi], 1)
    rg = np.random.default_rng(3)

    def rel(a, b):
        c, s_ = np.cos(a[2]), np.sin(a[2])
        return np.array([c * (b[0] - a[0]) + s_ * (b[1] - a[1]), -s_ * (b[0] - a[0]) + c * (b[1] - a[1]),
                         (b[2] - a[2] + np.pi) % (2 * np.pi) - np.pi])
    guess = np.zeros((nn, 3))
    guess[0] = tru[0]
    for i in range(1, nn):  # drifting odometry as the initial guess
        d = rel(tru[i - 1], tru[i]) + rg.normal(0, [0.002, 0.002, 0.0005])
        c, s_ = np.cos(guess[i - 1, 2]), np.sin(guess[i - 1, 2])
        guess[i] = [guess[i - 1, 0] + c * d[0] - s_ * d[1], guess[i - 1, 1] + s_ * d[0] + c * d[1], guess[i - 1, 2] + d[2]]
    pg = MPg.PoseGraph(lm_iterations=40, cg_iterations=2000)
    sv = pg.as_scan_solver()
    dp = C.POINTER(C.c_double)
    for i in range(nn):
        sv.add_node(sv.user, i, np.ascontiguousarray(guess[i]).ctypes.data_as(dp))
    cov = np.ascontiguousarray((np.eye(3) * [2.5e-4, 2.5e-4, 1e-5]).ravel())
    n_con = 0
    for i in range(nn):
        for j in ([i + 1, i + 2] + ([i - per_lap] if i >= per_lap and i % 5 == 0 else [])):
            if 0 <= j < nn and j != i:
                a, b = (i, j) if j > i else (j, i)
                d = np.ascontiguousarray(rel(tru[a], tru[b]) + rg.normal(0, [0.005, 0.005, 0.001]))
                sv.add_constraint(sv.user, a, b, d.ctypes.data_as(dp), cov.ctypes.data_as(dp))
                n_con += 1
    ids, outp = np.zeros(nn, np.int32), np.zeros((nn, 3))
    t0 = time.perf_counter()
    sv.compute(sv.user, nn, ids.ctypes.data_as(C.POINTER(C.c_int32)), outp.ctypes.data_as(dp))
    dt = time.perf_counter() - t0
    st = pg.stats()
    res = {"nodes": nn, "constraints": n_con, "solve_ms": dt * 1e3, "lm_steps": st["lm_steps"],
           "chi2_before": st["chi2_before"], "chi2_after": st["chi2_after"],
           "max_xy_err_before_m": float(np.abs(guess[:, :2] - tru[:, :2]).max()),
           "max_xy_err_after_m": float(np.abs(outp[:, :2] - tru[:, :2]).max()),
           "note": "host only (1 thread), first node fixed"}
    pg.close()
    return res


# ------------------------------------------------------------------------------------------------ workloads

def base_line(ctx, args, value, ms_max, steps, config, e2e, roofline, launches, clocks, scaling="weak", extra=None):
    line = {"metric": METRIC, "value": value, "unit": "scan-matches/s", "n_gpus": ctx.world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms_max / max(steps, 1), "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": config, "e2e": e2e,
            "gpu_launches": launches, "roofline": roofline, "clocks": clocks}
    if extra:
        line.update(extra)
    return line


def k1_roofline(sweep_ms, matches_per_launch, a1_bytes, clocks, traffic_key, batch):
    peak, peak_src = hbm_peak()
    traffic, traffic_src = committed_traffic(traffic_key, batch)
    sweep_ms = max(float(sweep_ms), 1e-6)
    achieved = a1_bytes * matches_per_launch / (sweep_ms * 1e-3) / 1e9
    sm_clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
    smem_ceiling = 148 * 32 * sm_clk  # 4-byte bank accesses / s
    lookups = a1_bytes * matches_per_launch / (sweep_ms * 1e-3)
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src, "kernel": "k_sweep_window", "kernel_ms": sweep_ms,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": a1_bytes * matches_per_launch,
            "note": "K1 is not DRAM-bound: the algorithmic bytes are served from shared memory (effective bandwidth, "
                    "hence frac > 1); see smem_gather for the resource that binds",
            "smem_gather": {"lookups_per_s": lookups, "bank_ceiling_per_s": smem_ceiling,
                            "frac_of_bank_ceiling": lookups / smem_ceiling,
                            "lookups_per_clk_per_sm": lookups / (148 * sm_clk)}}


def workload_cfg2(ctx, args, strong=False):
    torch, pkg = ctx.torch, ctx.pkg
    abi, synth = pkg.abi, pkg.synth
    M = pkg.load("matcher")
    world, rank, local = ctx.world, ctx.rank, ctx.local
    if strong:  # a FIXED total of args.batch matches split over the ranks
        from importlib import import_module
        par = import_module(PKG + ".parallel")
        lo, hi = par.shard_bounds(args.batch, world, rank)
        B = hi - lo
        allr = make_workload(synth, args.batch, 0)
        ranges, poses, bran, bpos = (a[lo:hi] for a in allr)
    else:
        B = args.batch
        ranges, poses, bran, bpos = make_workload(synth, B, rank)
    stream = ctx.stream
    params, laser = abi.matcher_params(1.5, 0.05, 0.03, 9.25), abi.laser_from(synth.Laser())
    m = M.ScanMatcher(params, laser, max_batch=B, max_base_scans=1, device=local, stream=stream.cuda_stream)
    se = abi.Search(0.75, 0.75, 0.05, 0.05, 22.5 * D, 0.25 * D, 1, 0)

    # ------------------------------------------------------------ resident-in-HBM arm ("value")
    m.set_scans(ranges, poses)
    m.add_scans(bran, bpos)
    m.sync()
    for _ in range(args.warmup):
        m.correlate_scan(poses, se)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    sweep_ms, lut_ms, red_ms = [], [], []
    last = {}

    def step():
        last["out"] = m.correlate_scan(poses, se)
        t = m.last_timing()
        sweep_ms.append(t["sweep_ms"]); lut_ms.append(t["lut_ms"]); red_ms.append(t["reduce_ms"])

    ms_max, per_rank_ms, steps_done = ctx.timed(step, args.steps, args.min_seconds)
    out = last["out"]
    assert (out[3] == 0).all() and m.last_timing()["path"] == 2
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    empty_frac = m.last_stats()["empty_window_frac"]
    total = (args.batch if strong else world * B)
    value = total * steps_done / (ms_max * 1e-3)

    # ------------------------------------------------------------ end-to-end arm (host buffers, pinned)
    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, C.cast(t.data_ptr(), C.POINTER(C.c_double))

    keep = [pinned(x) for x in (ranges, poses, bran, bpos)]
    pr, pp, pbr, pbp = (k[1] for k in keep)
    res = (abi.MatchResult * B)()
    L = M.lib()

    # two handles, two streams, a 2-deep pipeline: step i+1's uploads / rasterisation / lookup lists are enqueued before
    # step i's results are awaited, so they overlap step i's sweep.  Every step still uploads its own inputs from pinned
    # host memory and reads its own results back inside the timed region.
    stream2 = torch.cuda.Stream(device=local)
    m2 = M.ScanMatcher(params, laser, max_batch=B, max_base_scans=1, device=local, stream=stream2.cuda_stream)
    handles, results = [m.h, m2.h], [res, (abi.MatchResult * B)()]
    L.b2s_matcher_correlate_scan_begin.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(abi.Search), C.c_void_p]
    L.b2s_matcher_correlate_scan_end.argtypes = [C.c_void_p, C.POINTER(abi.MatchResult)]

    def e2e_begin(i):
        h = handles[i % 2]
        M.check(L.b2s_matcher_set_scans(h, B, pr, pp))
        M.check(L.b2s_matcher_add_scans(h, 1, pbr, pbp))
        M.check(L.b2s_matcher_correlate_scan_begin(h, pp, C.byref(se), None))

    def e2e_end(i):
        M.check(L.b2s_matcher_correlate_scan_end(handles[i % 2], results[i % 2]))

    def e2e_run(steps):
        e2e_begin(0)
        for i in range(steps):
            if i + 1 < steps:
                e2e_begin(i + 1)
            e2e_end(i)

    e2e_run(max(args.warmup, 2))
    ctx.barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    e2e_run(steps_done)
    e3.record(stream)  # every step's results have been awaited on the host: both streams are idle here
    ctx.barrier()
    e2e_ms = ctx.max_ms(e2.elapsed_time(e3))
    e2e_value = total * steps_done / (e2e_ms * 1e-3)
    h2d = int(ranges.nbytes + poses.nbytes + bran.nbytes + bpos.nbytes + poses.nbytes)
    d2h = int(C.sizeof(abi.MatchResult) * B)

    # ------------------------------------------------------------ the mapper-shaped variants of the same metric (rank 0, N = 1)
    variants = {}
    if world == 1 and not strong:
        try:
            m.set_kernel(3)  # sweep every beam (no empty-window dropping)
            for _ in range(2):
                m.correlate_scan(poses, se)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                m.correlate_scan(poses, se)
            torch.cuda.synchronize()
            variants["dense_no_window_skipping"] = {"matches_per_s": 3 * B / (time.perf_counter() - t0),
                                                    "sweep_ms": m.last_timing()["sweep_ms"]}
            m.set_kernel(0)
            # grids rasterised from a 70-scan running window (scan_buffer_size default), the mapper's shape
            nb_base, Bv = 70, 128
            _, tp, tr = synth.make_trajectory(77, nb_base + 1, synth.Laser(), step_xy=0.1, step_th_deg=3)
            mv = M.ScanMatcher(params, laser, max_batch=Bv, max_base_scans=nb_base, device=local, stream=stream.cuda_stream)
            vr = np.tile(tr[-1][None], (Bv, 1))
            vp = np.tile(tp[-1][None], (Bv, 1)) + np.random.default_rng(1).uniform(-0.05, 0.05, (Bv, 3))
            mv.set_scans(vr, vp)
            mv.add_scans(np.tile(tr[None, :nb_base], (Bv, 1, 1)), np.tile(tp[None, :nb_base], (Bv, 1, 1)))
            for _ in range(2):
                mv.correlate_scan(vp, se)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                ov = mv.correlate_scan(vp, se)
            torch.cuda.synchronize()
            variants["running_window_70_base_scans"] = {"batch": Bv, "matches_per_s": 3 * Bv / (time.perf_counter() - t0),
                                                        "sweep_ms": mv.last_timing()["sweep_ms"],
                                                        "empty_window_frac": mv.last_stats()["empty_window_frac"],
                                                        "ok": int((ov[3] == 0).sum())}
            mv.close()
        except Exception as e:
            variants["error"] = repr(e)
    sampler.stop()
    clocks = sampler.summary()
    sweep = float(np.mean(sweep_ms))
    line = None
    if rank == 0:
        cfg = cfg2_config(B, world)
        if strong:
            cfg = dict(cfg, workload="strong", total_matches=args.batch, parallelism=f"a fixed {args.batch}-match batch split x{world}")
        line = base_line(
            ctx, args, value, ms_max, steps_done, cfg,
            {"value": e2e_value, "unit": "scan-matches/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
             "includes": "set_scans + add_scans (rasterise) + correlate_scan_begin/_end from pinned host buffers, "
                         "2-deep pipeline over two handles (each step uploads its inputs and reads its results back)"},
            k1_roofline(sweep, B, A1_BYTES, clocks, "k_sweep_window", B), steps_done * KERNELS_PER_STEP, clocks,
            scaling="strong" if strong else "weak",
            extra={"stage_ms": {"lut": float(np.mean(lut_ms)), "sweep": sweep, "reduce": float(np.mean(red_ms))},
                   "per_rank_ms_per_step": [x / steps_done for x in per_rank_ms],
                   "timed_seconds": ms_max * 1e-3,
                   "empty_windows_dropped": {"frac_of_beam_angle_pairs": empty_frac,
                                             "note": "beams whose whole 31x31 window lies in empty 4x4 grid blocks add 0 to every "
                                                     "candidate and are dropped when the sorted lists are built; the response volume "
                                                     "is bit-identical (tests/test_gpu_matcher.py compares every candidate); "
                                                     "b2s_matcher_set_kernel(m, 3) sweeps every beam (variants.dense_no_window_skipping)"},
                   "variants": variants})
        line["multi_gpu_exact"] = oracle_check_matches(pkg, params, laser, ranges, poses, bran, bpos, se, out, [0, B - 1])
        if world == 1 and not strong and not args.no_k2:
            try:
                line["grid_cells"], line["roofline_k2"] = bench_k2(pkg, local, args.quick)
                line["grid_cells"]["cfg5_pose_graph_solve_cpu"] = pose_graph_solve(pkg, 1000 if args.quick else 5000)
            except Exception as e:  # the headline metric must not be lost to a secondary one
                line["grid_cells"] = {"error": repr(e)}
        if world == 1 and not strong and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(pkg, min(args.cpu_sample, B), ranges, poses, bran, bpos)
    m.close()
    m2.close()
    return line


def workload_cfg4(ctx, args):
    """BASELINE cfg 4: correlative search-window sweep 11x11x61 -> 61x61x361 on a 0.025 m grid, batch-sharded."""
    torch, pkg = ctx.torch, ctx.pkg
    abi, synth = pkg.abi, pkg.synth
    M = pkg.load("matcher")
    world, rank, local = ctx.world, ctx.rank, ctx.local
    l4 = synth.Laser(range_threshold=9.25)
    params, laser = abi.matcher_params(1.5, 0.025, 0.03, 9.25), abi.laser_from(l4)
    B4 = 64 if args.quick else 256
    cases = [synth.make_match_case(4_000_000 + rank * B4 + i, l4) for i in range(B4)]
    mr, mp = np.stack([c.ranges for c in cases]), np.stack([c.odom_pose for c in cases])
    mbr, mbp = np.stack([c.base_ranges for c in cases])[:, None, :], np.stack([c.base_pose for c in cases])[:, None, :]
    m4 = M.ScanMatcher(params, laser, max_batch=B4, max_base_scans=1, device=local, stream=ctx.stream.cuda_stream)
    m4.set_scans(mr, mp)
    m4.add_scans(mbr, mbp)
    sampler = ClockSampler(local)
    sampler.start()
    rows, head = [], None
    for W, nth, sub in ((11, 61, B4), (31, 181, B4), (61, 361, max(8, B4 // 8))):
        half = 0.5 * (W - 1) * 0.025
        se4 = abi.Search(half, half, 0.025, 0.025, 0.5 * (nth - 1) * 0.25 * D, 0.25 * D, 1, 0)
        if sub != B4:
            m4.set_scans(mr[:sub], mp[:sub])
            m4.add_scans(mbr[:sub], mbp[:sub])
        for _ in range(max(args.warmup, 1)):
            r4 = m4.correlate_scan(mp[:sub], se4)
        sw = []

        def step():
            m4.correlate_scan(mp[:sub], se4)
            sw.append(m4.last_timing()["sweep_ms"])
        ms_max, per_rank, done = ctx.timed(step, max(2, args.steps // (1 if W < 61 else 4)), args.min_seconds)
        row = {"window": [W, W, nth], "batch_per_gpu": sub, "matches_per_s": world * sub * done / (ms_max * 1e-3),
               "ms_per_step": ms_max / done, "sweep_ms": float(np.mean(sw)), "path": m4.last_timing()["path"],
               "lookups_per_s_kernel": world * sub * W * W * nth * 1081 / (float(np.mean(sw)) * 1e-3),
               "ok": int((r4[3] == 0).sum()), "per_rank_ms_per_step": [x / done for x in per_rank]}
        if W == 11:
            row["multi_gpu_exact"] = oracle_check_matches(pkg, params, laser, mr, mp, mbr, mbp, se4, r4, [0, 1])
        rows.append(row)
        if W == 31:
            head = (row, ms_max, done, float(np.mean(sw)), sub)
    sampler.stop()
    clocks = sampler.summary()
    m4.close()
    if rank != 0:
        return None
    row, ms_max, done, sweep, sub = head
    a1 = 31 * 31 * 181 * 1081
    cfg = {"workload": "cfg4", "grid_res_m": 0.025, "grid": "807 x 807 cells (652 KB, 4 row bands in shared memory)", "beams": NBEAMS,
           "windows": [[11, 11, 61], [31, 31, 181], [61, 61, 361]], "value_window": [31, 31, 181],
           "batch_per_gpu": sub, "parallelism": f"batch-shard x{world}",
           "l2_policy": f"inputs larger than L2 ({sub} grids x 652 KB + {sub * 181 * 961 * 4 / 1e6:.0f} MB volume per step)"}
    return base_line(ctx, args, row["matches_per_s"], ms_max, done, cfg,
                     {"value": None, "unit": "scan-matches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                      "note": "cfg4 is measured resident-in-HBM only; the end-to-end arm is the cfg2 line"},
                     k1_roofline(sweep, sub, a1, clocks, "k_sweep_window_cfg4", sub), done * KERNELS_PER_STEP, clocks,
                     extra={"rows": rows, "multi_gpu_exact": rows[0].get("multi_gpu_exact")})


def workload_cfg5(ctx, args):
    """BASELINE cfg 5: a many-lap trajectory through b2s_mapper with the lesson6 outdoor yaml; the loop-closure candidate
    chains its TryCloseLoop examines (logged through the matcher plug-in while the real CUDA matcher answers) are then
    replayed as ONE batch-sharded coarse MatchScan job list over the ranks; then the CPU pose-graph solve."""
    torch, pkg = ctx.torch, ctx.pkg
    abi, synth = pkg.abi, pkg.synth
    M, MPm = pkg.load("matcher"), pkg.load("mapper")
    world, rank, local = ctx.world, ctx.rank, ctx.local
    n_nodes = 300 if args.quick else args.nodes
    lo_ = synth.Laser(range_threshold=50.0)
    # outdoor yaml (lesson6/config/mapper_params_outdoor.yaml); penalties squared / converted as setParam* does
    yaml = dict(scan_buffer_size=110, scan_buffer_maximum_scan_distance=50.0, link_match_minimum_response_fine=0.1,
                link_scan_maximum_distance=1.5, loop_search_maximum_distance=15.0, loop_match_minimum_chain_size=5,
                loop_match_maximum_variance_coarse=9.0, loop_match_minimum_response_coarse=0.35,
                loop_match_minimum_response_fine=0.45, minimum_travel_heading=0.174,
                sequential_search_size=0.3, sequential_resolution=0.05, sequential_smear_deviation=0.03,
                loop_search_size=15.0, loop_resolution=0.1, loop_smear_deviation=0.3,
                both_distance_variance_penalty=0.09, both_angle_variance_penalty=0.01,
                both_fine_search_angle_offset=0.00349, both_coarse_search_angle_offset=0.349,
                both_coarse_angle_resolution=0.0349, both_use_response_expansion=1)
    prm = MPm.default_params(50.0, **yaml)
    al = abi.laser_from(lo_)
    # every rank enumerates redundantly (deterministic inputs, own GPU): no broadcast of megabytes of chains needed
    _, tru, odo, rng_m = synth.make_loop_trajectory(23, n_nodes, lo_, radius=12.0, step=0.5, half_w=30.0, half_h=22.0, n_boxes=14)
    handles = {}
    jobs = []  # (ranges, pose, base_ranges[nb, N], base_poses[nb, 3])

    def match_fn(user, which, batch, ranges, poses, base_first, n_base, base_ranges, base_poses, do_pen, do_ref, results):
        try:
            N = al.n_readings
            nb = [n_base[b] for b in range(batch)]
            mx = max(max(nb), 1)
            key = (which,)
            if key not in handles or handles[key].max_batch < batch or handles[key].cap_base < mx:
                if key in handles:
                    handles[key].close()
                h = M.ScanMatcher(prm.loop if which else prm.sequential, al, max_batch=max(batch, 8), max_base_scans=max(mx, 128),
                                  device=local)
                h.cap_base = max(mx, 128)
                handles[key] = h
            h = handles[key]
            total = sum(nb)
            r = np.ctypeslib.as_array(ranges, shape=(batch, N)).copy()
            p = np.ctypeslib.as_array(poses, shape=(batch, 3)).copy()
            br_all = np.ctypeslib.as_array(base_ranges, shape=(max(total, 1), N))
            bp_all = np.ctypeslib.as_array(base_poses, shape=(max(total, 1), 3))
            br = np.zeros((batch, mx, N)); bp = np.zeros((batch, mx, 3))
            for b in range(batch):
                f = base_first[b]
                if nb[b] == 0:
                    continue
                br[b, :nb[b]] = br_all[f:f + nb[b]]; bp[b, :nb[b]] = bp_all[f:f + nb[b]]
                br[b, nb[b]:] = br_all[f]; bp[b, nb[b]:] = bp_all[f]  # pad by repeating a base scan (max-stamp: no change)
                if which == 1 and rank_log[0]:
                    seen[0] += 1
                    if len(jobs) < 1024:  # the replay set is bounded (each chain carries up to ~0.7 MB of readings)
                        jobs.append((r[b].copy(), p[b].copy(), br_all[f:f + nb[b]].copy(), bp_all[f:f + nb[b]].copy()))
            out = h.match_scan_host(r, p, br, bp, bool(do_pen), bool(do_ref))
            for b in range(batch):
                cv = out[2][b]
                # Two qualifying cells on a diagonal of the coarse lattice make xx * yy == xy^2: the reference's
                # Matrix3::Inverse asserts on such a link covariance (and so does b2s_mapper_process).  The enumeration pass
                # conditions those (counted) so that the synthetic trajectory can be walked to its end.
                if out[3][b] == 0 and abs(cv[0, 0] * cv[1, 1] - cv[0, 1] * cv[1, 0]) <= 1e-9 * abs(cv[0, 0] * cv[1, 1]):
                    cv[0, 1] *= 0.98; cv[1, 0] *= 0.98
                    conditioned[0] += 1
                results[b].response = out[0][b]
                for i in range(3):
                    results[b].pose[i] = out[1][b][i]
                for i in range(9):
                    results[b].cov[i] = out[2][b].ravel()[i]
                results[b].status = int(out[3][b]); results[b].tie_count = int(out[4][b])
            return 0
        except Exception as e:  # never let an exception cross the C boundary
            sys.stderr.write(f"cfg5 match_fn: {e!r}\n")
            return 4

    rank_log = [True]
    conditioned = [0]
    seen = [0]
    pg = MPm.PoseGraph(lm_iterations=40, cg_iterations=400)
    mapper = MPm.Mapper(prm, al, device=local, match_fn=match_fn)
    mapper.set_scan_solver(pg.as_scan_solver())
    t0 = time.perf_counter()
    for i in range(n_nodes):
        mapper.process(rng_m[i], odo[i], 0.1 * i)
    t_map = time.perf_counter() - t0
    stm = mapper.stats()
    n_edges = int(len(mapper.edges()[0]))
    err = float(np.abs(mapper.poses()[:, :2] - tru[:len(mapper.poses()), :2]).max())
    mapper.close()
    for h in handles.values():
        h.close()
    # ---- the replay: all logged loop-closure candidate chains, sharded round-robin over the ranks, coarse MatchScan
    mine = jobs[rank::world]
    nj = len(mine)
    sampler = ClockSampler(local)
    sampler.start()
    value, ms_max, done, sweep, row = 0.0, 1.0, 0, 1.0, {}
    if len(jobs) >= world and nj > 0:
        mxb = max(len(j[2]) for j in jobs)
        Bc = min(64, nj)
        hl = M.ScanMatcher(prm.loop, al, max_batch=Bc, max_base_scans=mxb, device=local, stream=ctx.stream.cuda_stream)
        N = al.n_readings

        def pack(chunk):
            r = np.stack([j[0] for j in chunk]); p = np.stack([j[1] for j in chunk])
            br = np.zeros((len(chunk), mxb, N)); bp = np.zeros((len(chunk), mxb, 3))
            for b, j in enumerate(chunk):
                k = len(j[2])
                br[b, :k] = j[2]; bp[b, :k] = j[3]
                br[b, k:] = j[2][0]; bp[b, k:] = j[3][0]
            return r, p, br, bp
        chunks = [pack(mine[i:i + Bc]) for i in range(0, nj, Bc)]
        results = []

        def step():
            results.clear()
            for r, p, br, bp in chunks:
                results.append(hl.match_scan_host(r, p, br, bp, False, False))  # TryCloseLoop: coarse only, no penalty
        for _ in range(max(1, args.warmup // 2)):
            step()
        ms_max, per_rank, done = ctx.timed(step, max(1, args.steps // 3), args.min_seconds)
        sweep = hl.last_timing()["sweep_ms"]
        accepted = int(sum(((o[0] > prm.loop_match_minimum_response_coarse) & (o[3] == 0)).sum() for o in results))
        value = len(jobs) * done / (ms_max * 1e-3)
        row = {"candidate_chains": len(jobs), "candidate_chains_seen_by_the_mapper": seen[0], "chains_this_rank": nj, "max_chain": mxb, "batch": Bc,
               "coarse_accepted_this_rank": accepted, "per_rank_ms_per_step": [x / done for x in per_rank],
               "path": hl.last_timing()["path"]}
        hl.close()
    sampler.stop()
    clocks = sampler.summary()
    if rank != 0:
        pg.close()
        return None
    # ---- the CPU solve of the graph the mapper built (re-run of Compute on the final graph)
    sv = pg.as_scan_solver()
    nn = stm["running_scans"]
    ids, outp = np.zeros(max(n_nodes, 1), np.int32), np.zeros((max(n_nodes, 1), 3))
    t0 = time.perf_counter()
    sv.compute(sv.user, n_nodes, ids.ctypes.data_as(C.POINTER(C.c_int32)), outp.ctypes.data_as(C.POINTER(C.c_double)))
    t_solve = time.perf_counter() - t0
    stg = pg.stats()
    pg.close()
    cfg = {"workload": "cfg5", "key_frames": n_nodes, "yaml": "lesson6/config/mapper_params_outdoor.yaml", "beams": NBEAMS,
           "loop_matcher": "15 m / 0.1 m, smear 0.3: 1165 x 1168 B grid (1.36 MB), coarse 76x76x21 every other cell",
           "parallelism": f"candidate chains sharded round-robin x{world}", "l2_policy": "each step re-uploads and re-rasterises every chain"}
    a1 = 76 * 76 * 21 * 1081
    return base_line(ctx, args, value, ms_max, done, cfg,
                     {"value": value, "unit": "scan-matches/s", "h2d_bytes_per_step": int(sum(j[2].nbytes + j[0].nbytes for j in mine)),
                      "d2h_bytes_per_step": nj * 112, "note": "the replay goes through b2s_matcher_match_scan_host (host buffers in, "
                      "results out), so value IS the end-to-end number"},
                     k1_roofline(sweep, min(64, max(nj, 1)), a1, clocks, "k_sweep_window_cfg5", None), done * 8, clocks,
                     extra={"metric": "loop-closure candidate scan-matches/s (coarse MatchScan 76x76x21, 1081 beams)",
                            "replay": row,
                            "mapper": {"seconds": t_map, "key_frames_per_s": n_nodes / t_map, "match_scan_calls": stm["match_calls"],
                                       "loop_candidates": stm["loop_candidates"], "loops_closed": stm["loops_closed"],
                                       "edges": n_edges, "max_xy_err_m": err, "singular_covariances_conditioned": conditioned[0],
                                       "note": "enumeration pass through the Python matcher plug-in (untimed for the metric)"},
                            "pose_graph_solve_cpu": {"nodes": stg["nodes"], "constraints": stg["constraints"], "solve_ms": t_solve * 1e3,
                                                     "lm_steps": stg["lm_steps"], "chi2_before": stg["chi2_before"],
                                                     "chi2_after": stg["chi2_after"]}})


def workload_k2(ctx, args):
    sections, roof = bench_k2(ctx.pkg, ctx.local, args.quick)
    if ctx.rank != 0:
        return None
    v = sections.get("hector_batched_maps", {}).get("cells_per_s", 0.0)
    return {"metric": "grid cells/s (Bresenham cell visits, batched Hector maps)", "value": v, "unit": "cells/s", "n_gpus": ctx.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 log-odds / u32 counters", "data": "synthetic", "config": {"workload": "k2"},
            "e2e": {"value": sections.get("hector_stream", {}).get("stream_exact", {}).get("cells_per_s"), "unit": "cells/s",
                    "h2d_bytes_per_step": sections.get("hector_stream", {}).get("stream_exact", {}).get("h2d_bytes"),
                    "d2h_bytes_per_step": sections.get("hector_stream", {}).get("stream_exact", {}).get("d2h_bytes")},
            "gpu_launches": 3 * 21, "roofline": roof.get("hector_batched_maps"), "roofline_k2": roof, "grid_cells": sections}


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner at
    NCCL_DEBUG=VERSION / WARN, and whole pages at INFO), so file descriptor 1 is pointed at stderr for the run and the
    line goes out through a private duplicate of the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
        return
    sys.stdout.flush()
    while data:
        data = data[os.write(_REAL_STDOUT, data):]


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    ctx = Ctx(args)
    if args.workload == "cfg2":
        line = workload_cfg2(ctx, args)
    elif args.workload == "strong":
        line = workload_cfg2(ctx, args, strong=True)
    elif args.workload == "cfg4":
        line = workload_cfg4(ctx, args)
    elif args.workload == "cfg5":
        line = workload_cfg5(ctx, args)
    else:
        line = workload_k2(ctx, args)
    if ctx.rank == 0 and line is not None:
        emit(line)
    ctx.close()


if __name__ == "__main__":
    main()
