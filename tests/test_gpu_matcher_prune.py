"""GPU tests for angle pruning in the K1 window sweep (k_prune_select).

Kernel selector 2 (like 0) bounds every (angle, 4x4 candidate block) from a max-pooled grid and sweeps only the angles
that can hold the best response, a tie or a per-cell maximum the covariance reads; selector 3 sweeps every beam and
every angle.  Every output must be bit-identical between the two.
"""
import numpy as np
import pytest

from oracle import port

pytestmark = pytest.mark.gpu
D = 0.01745329251994329577


@pytest.fixture(scope="module")
def M(pkg):
    m = pkg.load("matcher")
    assert m.device_count() > 0, "no CUDA device: the product path has no fallback"
    return m


def cfg2(abi, synth):
    params, laser = abi.matcher_params(1.5, 0.05, 0.03, 9.25), abi.laser_from(synth.Laser())
    return params, laser


def search(abi, pen=1):
    return abi.Search(0.75, 0.75, 0.05, 0.05, 22.5 * D, 0.25 * D, pen, 0)


def cases(synth, seeds):
    cs = [synth.make_match_case(s, dropout=0.03 if s % 4 == 3 else 0.0) for s in seeds]
    ranges = np.stack([c.ranges for c in cs])
    ranges[1::8, ::17] = np.nan
    ranges[2::8, 5::29] = np.inf
    return (ranges, np.stack([c.odom_pose for c in cs]), np.stack([c.base_ranges for c in cs])[:, None, :],
            np.stack([c.base_pose for c in cs])[:, None, :])


def both(m, centers, se):
    """(pruned, dense) results of one CorrelateScan, and the pruned call's prune statistics."""
    m.set_kernel(2)
    pruned = m.correlate_scan(centers, se)
    assert m.last_timing()["path"] == 2
    stats = m.last_prune_stats()
    m.set_kernel(3)
    dense = m.correlate_scan(centers, se)
    m.set_kernel(0)
    return pruned, dense, stats


def assert_same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("pen", [1, 0])
def test_pruned_equals_dense_cfg2(pkg, M, pen):
    """64 seeded cfg2 matches (NaN / inf dropouts included): response, pose, covariance, status and tie count equal the
    dense sweep's; the seeds include matches whose top-bound block does not hold the best response."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    ranges, poses, bran, bpos = cases(synth, range(1_000_000, 1_000_064))
    B = len(ranges)
    m = M.ScanMatcher(params, laser, max_batch=B, max_base_scans=1)
    m.set_scans(ranges, poses)
    m.add_scans(bran, bpos)
    pruned, dense, st = both(m, poses, search(abi, pen))
    assert (dense[3] == 0).all()
    assert_same(pruned, dense)
    if pen:
        assert st["kept_frac"] < 0.5, st
    assert 0 < st["swept"] <= B * 181
    assert m.last_prune_stats() == {"kept_frac": 1.0, "swept": B * 181}  # selector 3: nothing pruned
    m.close()


def test_response_sums_after_pruned_sweep(pkg, M):
    """After a pruned sweep the exported volume is still the whole volume (swept densely on demand)."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    ranges, poses, bran, bpos = cases(synth, range(1_000_000, 1_000_004))
    m = M.ScanMatcher(params, laser, max_batch=4, max_base_scans=1)
    m.set_scans(ranges, poses)
    m.add_scans(bran, bpos)
    se = search(abi)
    m.correlate_scan(poses, se)
    assert m.last_prune_stats()["kept_frac"] < 0.5
    for b in (0, 3):
        pm = port.PortMatcher(params, laser)
        pm.set_scan(ranges[b], poses[b])
        pm.add_scans(bran[b], bpos[b])
        pm.correlate_scan(pm.sp, se, want_sums=True)
        assert np.array_equal(m.response_sums(b, (31, 31, 181)), pm.last_sums)
    m.close()


def test_empty_grid_nothing_pruned(pkg, M):
    """No base scans: every candidate ties at response 0, so no angle may be pruned."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    ranges, poses, _, _ = cases(synth, range(10, 12))
    m = M.ScanMatcher(params, laser, max_batch=2, max_base_scans=1)
    m.set_scans(ranges, poses)
    m.add_scans(np.zeros((2, 0, 1081)), np.zeros((2, 0, 3)))
    pruned, dense, st = both(m, poses, search(abi))
    assert_same(pruned, dense)
    assert st["kept_frac"] == 1.0
    assert (dense[4] == 31 * 31 * 181).all()
    m.close()


def test_two_peaks_at_distant_angles(pkg, M):
    """The base scan rasterised twice, the second copy turned by 0.3 rad about its sensor: two near-equal peaks far
    apart in angle, both kept."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    cs = [synth.make_match_case(s, max_xy=0.02, max_th_deg=1.0) for s in range(2000, 2004)]
    ranges, poses = np.stack([c.ranges for c in cs]), np.stack([c.odom_pose for c in cs])
    bran2 = np.stack([np.stack([c.base_ranges, c.base_ranges]) for c in cs])
    bpos2 = np.stack([np.stack([c.base_pose, c.base_pose]) for c in cs])
    bpos2[:, 1, 2] += 0.3
    centers = poses.copy()
    centers[:, 2] += 0.15  # midway between the two copies: peaks near -0.15 and +0.15 rad of the +-0.39 rad window
    m = M.ScanMatcher(params, laser, max_batch=4, max_base_scans=2)
    m.set_scans(ranges, poses)
    m.add_scans(bran2, bpos2)
    pruned, dense, st = both(m, centers, search(abi))
    assert_same(pruned, dense)
    assert st["swept"] < 4 * 181
    m.close()


def test_out_of_range_lattice(pkg, M):
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    ranges, poses, bran, bpos = cases(synth, range(3000, 3003))
    m = M.ScanMatcher(params, laser, max_batch=3, max_base_scans=1)
    m.set_scans(ranges, poses)
    m.add_scans(bran, bpos)
    centers = poses.copy()
    centers[1, 0] += 50.0
    pruned, dense, _ = both(m, centers, search(abi))
    assert_same(pruned, dense)
    assert pruned[3][1] == abi.B2S_ERR_OUT_OF_RANGE and pruned[3][0] == pruned[3][2] == abi.B2S_OK
    m.close()


def lattice_irregular(cx, cy, gox, goy):
    """k_bases's test on the host: is the candidate lattice NOT the raster base00 + (ix + iy * width_step)?"""
    scale = 1.0 / 0.05

    def w2g(w, o):
        v = (w - o) * scale
        return np.copysign(np.floor(np.abs(v) + 0.5), v)

    k = np.arange(31, dtype=np.float64)
    gx = w2g(cx + (-0.75 + k * 0.05), gox)
    gy = w2g(cy + (-0.75 + k * 0.05), goy)
    return bool((gx != gx[0] + np.arange(31)).any() or (gy != gy[0] + np.arange(31)).any())


def test_irregular_lattice_falls_through(pkg, M):
    """A search centre on a rounding tie of the grid: the lattice is not the regular raster, the match goes to the
    generic kernel and keeps every angle, its neighbours are pruned."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    ranges, poses, bran, bpos = cases(synth, range(4000, 4003))
    m = M.ScanMatcher(params, laser, max_batch=3, max_base_scans=1)
    m.set_scans(ranges, poses)
    m.add_scans(bran, bpos)
    gox, goy = m.grid(1)[1]
    centers = poses.copy()
    found = False
    tie = gox + (np.floor((poses[1, 0] - gox) / 0.05) + 0.5) * 0.05
    lo = hi = tie
    for _ in range(4000):  # walk outwards from the tie one ulp at a time
        for cx in (lo, hi):
            if lattice_irregular(cx, centers[1, 1], gox, goy):
                centers[1, 0] = cx
                found = True
                break
        if found:
            break
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
    assert found, "no centre on a rounding tie found"
    pruned, dense, st = both(m, centers, search(abi))
    assert_same(pruned, dense)
    assert 181 < st["swept"] < 3 * 181
    m.close()


def test_begin_end_pipelined_pruned(pkg, M):
    """correlate_scan_begin/_end interleaved over two handles (pruned) equal the synchronous dense sweep."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    se = search(abi)
    sets = [cases(synth, range(5000 + 10 * k, 5006 + 10 * k)) for k in range(4)]
    ms = [M.ScanMatcher(params, laser, max_batch=6, max_base_scans=1) for _ in range(2)]
    want = []
    ms[0].set_kernel(3)
    for r, p, br, bp in sets:
        ms[0].set_scans(r, p); ms[0].add_scans(br, bp)
        want.append(ms[0].correlate_scan(p, se))
    ms[0].set_kernel(0)

    def begin(i):
        r, p, br, bp = sets[i]
        ms[i % 2].set_scans(r, p); ms[i % 2].add_scans(br, bp); ms[i % 2].correlate_scan_begin(p, se)

    got = []
    begin(0)
    for i in range(4):
        if i + 1 < 4:
            begin(i + 1)
        got.append(ms[i % 2].correlate_scan_end())
        assert ms[i % 2].last_prune_stats()["kept_frac"] < 0.5
    for w, g in zip(want, got):
        assert_same(w, g)
    for m in ms:
        m.close()


def test_tiled_1024_identical(pkg, M):
    """1024 copies of one input give 1024 identical outputs, equal to the dense sweep of the same input."""
    abi, synth = pkg.abi, pkg.synth
    params, laser = cfg2(abi, synth)
    ranges, poses, bran, bpos = cases(synth, [1_000_005])
    B = 1024
    tile = lambda a: np.repeat(a, B, axis=0)
    m = M.ScanMatcher(params, laser, max_batch=B, max_base_scans=1)
    m.set_scans(tile(ranges), tile(poses))
    m.add_scans(tile(bran), tile(bpos))
    pruned, dense, st = both(m, tile(poses), search(abi))
    assert_same(pruned, dense)
    for a in pruned:
        assert (a == a[:1]).all()
    assert st["swept"] % B == 0 and st["kept_frac"] < 0.5
    m.close()
