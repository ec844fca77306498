"""GPU edge cases the reference's own call sites exercise: empty / NaN / gated clouds, points outside the map, sentinel
returns of the per-call API, and a local update box (SetUpdateRange)."""
import numpy as np
import pytest

from tests import scenes
from tests.parity import compare, invariants

pytestmark = pytest.mark.gpu


def pair(oracle_built, mode, origin=(-3.2, -3.2, -1.6), res=0.1, size=(6.4, 6.4, 3.2), params=scenes.PARAMS_DEFAULT):
    import fiesta_b200
    dev = fiesta_b200.ESDFMap(origin, res, size, mode=mode)
    ora = oracle_built.OracleMap(origin, res, size)
    dev.SetParameters(*params)
    ora.SetParameters(*params)
    return dev, ora


def same_counters(dev, ora):
    (h1, t1), (h2, t2) = dev.export_counters(), ora.export_counters()
    return np.array_equal(h1, h2) and np.array_equal(t1, t2)


@pytest.mark.parametrize("mode", ["fast", "exact"])
def test_degenerate_clouds(oracle_built, mode):
    dev, ora = pair(oracle_built, mode)
    T = scenes.body_transform((0.013, -0.021, 0.009), 0.3)
    rng = np.random.default_rng(0)
    clouds = [
        np.empty((0, 3), np.float32),                                            # empty frame
        np.full((100, 3), np.nan, np.float32),                                   # all NaN (Fiesta.h:202)
        (rng.normal(size=(500, 3)) * 0.1).astype(np.float32),                    # all shorter than min_ray_length (:209)
        (rng.normal(size=(2000, 3)) * 20).astype(np.float32),                    # mostly far outside the map / clipped (:211-213)
        np.tile(np.array([[1.0, 0.5, 0.2]], np.float32), (300, 1)),              # 300 identical points: endpoint dedupe (:227-230)
        (rng.normal(size=(3000, 3)) * 1.5).astype(np.float32),
    ]
    for k, pts in enumerate(clouds):
        assert dev.RaycastFrame(pts, T, 0.5, 5.0) == ora.RaycastFrame(pts, T, 0.5, 5.0), k
        assert same_counters(dev, ora), k
        assert dev.CheckUpdate() == ora.CheckUpdate(), k
        if dev.CheckUpdate():
            assert dev.UpdateOccupancy(True) == ora.UpdateOccupancy(True)
            dev.UpdateESDF(); ora.UpdateESDF()
        r = compare(dev, ora)
        assert r["occ"] == 0, (k, r)
        if mode == "exact":
            assert r["dist"] == 0 and r["cobs_tie"] == 0 and r["cobs_nontie"] == 0, (k, r)
    assert dev.stats()["rays_dropped"] == ora.hung_rays()


def test_per_call_api_and_sentinels(oracle_built):
    """int SetOccupancy(pos|vox, occ) return values and queries (ESDFMap.cpp:401-437, 452-540), call by call."""
    dev, ora = pair(oracle_built, "exact", params=scenes.PARAMS_TOGGLE)
    rng = np.random.default_rng(1)
    for _ in range(3000):
        p = rng.uniform(-3.6, 3.6, 3) * (1, 1, 0.55)
        occ = int(rng.integers(0, 3))                                            # 2 is invalid -> -10000
        assert dev.SetOccupancy(tuple(p), occ) == ora.SetOccupancy(tuple(p), occ)
    for _ in range(500):
        v = tuple(int(x) for x in rng.integers(0, 32, 3))
        occ = int(rng.integers(0, 2))
        assert dev.SetOccupancy(v, occ) == ora.SetOccupancy(v, occ)
    edge = (3.2, 3.2, 1.6)                                                       # exactly on the upper face: in map, voxel index aliases
    assert dev.SetOccupancy(edge, 1) == ora.SetOccupancy(edge, 1)
    assert same_counters(dev, ora)
    assert dev.UpdateOccupancy(True) == ora.UpdateOccupancy(True)
    dev.UpdateESDF(); ora.UpdateESDF()
    r = compare(dev, ora)
    assert r["dist"] == 0 and r["cobs_tie"] == 0 and r["occ"] == 0, r
    for _ in range(300):
        p = tuple(rng.uniform(-3.6, 3.6, 3) * (1, 1, 0.55))
        assert dev.GetDistance(p) == ora.GetDistance(p)
        assert dev.GetOccupancy(p) == ora.GetOccupancy(p)
        d1, g1 = dev.GetDistWithGradTrilinear(p)
        d2, g2 = ora.GetDistWithGradTrilinear(p)
        inside = all(-3.1 < p[i] < (3.0, 3.0, 1.4)[i] for i in range(3))
        if inside or d2 == -1:
            assert d1 == d2 and np.array_equal(g1, g2), p
    v = (5, 6, 7)
    assert dev.GetDistance(v) == ora.GetDistance(v) and dev.GetOccupancy(v) == ora.GetOccupancy(v)


@pytest.mark.parametrize("mode", ["fast", "exact"])
def test_local_update_box(oracle_built, mode):
    """SetUpdateRange (ESDFMap.cpp:792-810): observations outside the box are not counted and the wave stays inside it."""
    dev, ora = pair(oracle_built, mode, params=scenes.PARAMS_TOGGLE)
    allv = scenes.all_voxels(dev.grid_size)
    for m in (dev, ora):
        m.SetOccupancyBatchVox(allv, np.zeros(len(allv), np.uint8)); m.UpdateOccupancy(True); m.UpdateESDF()
    rng = np.random.default_rng(2)
    lo, hi = (-1.5, -1.0, -0.8), (1.2, 1.9, 0.9)
    for r in range(3):
        for m in (dev, ora):
            m.SetUpdateRange(lo, hi)
        vox = np.stack([rng.integers(0, dev.grid_size[i], 1500) for i in range(3)], -1).astype(np.int32)
        occ = (rng.random(1500) < 0.5).astype(np.uint8)
        assert np.array_equal(dev.SetOccupancyBatchVox(vox, occ), ora.SetOccupancyBatchVox(vox, occ))
        assert same_counters(dev, ora)
        assert dev.UpdateOccupancy(True) == ora.UpdateOccupancy(True)
        dev.UpdateESDF(); ora.UpdateESDF()
        res = compare(dev, ora)
        assert res["occ"] == 0 and res["dist"] == 0 and res["cobs_nontie"] == 0, (r, res)
        if mode == "exact":
            assert res["cobs_tie"] == 0, (r, res)
    for m in (dev, ora):
        m.SetOriginalRange()


def test_local_map_moving_box_exact(oracle_built):
    """Local-map mode (Fiesta.h:509-513 with global_update_ = false): a sliding update box + UpdateOccupancy(false).  A voxel
    observed outside the PREVIOUS box is reset to occupancy 0 / distance +infinity_ while its closest obstacle and its place in
    that obstacle's dependant list are kept (ESDFMap.cpp:256-259); the order-exact mode reproduces that state and everything
    that follows from it (arrays compared after every update)."""
    dev, ora = pair(oracle_built, "exact", params=scenes.PARAMS_TOGGLE)
    allv = scenes.all_voxels(dev.grid_size)
    rng = np.random.default_rng(7)
    idx = rng.choice(len(allv), 300, replace=False)
    for m in (dev, ora):                                        # every voxel observed, 300 obstacles: finite distances everywhere
        m.SetOccupancyBatchVox(allv, np.zeros(len(allv), np.uint8)); m.UpdateOccupancy(True); m.UpdateESDF()
        m.SetOccupancyBatchVox(allv[idx], np.ones(300, np.uint8)); m.UpdateOccupancy(True); m.UpdateESDF()
        m.SetParameters(*scenes.PARAMS_DEFAULT)                 # from here on one miss no longer clamps: resets are not skipped (:250-255)
    seen_reset = 0
    for r in range(8):
        c = np.array([-1.2 + 0.35 * r, -0.9 + 0.3 * r, 0.0])                       # the box slides through the map
        lo, hi = c - np.array([1.3, 1.2, 0.9]), c + np.array([1.3, 1.2, 0.9])
        for m in (dev, ora):
            m.SetUpdateRange(lo, hi)
        vox = np.stack([rng.integers(0, dev.grid_size[i], 6000) for i in range(3)], -1).astype(np.int32)
        occ = (rng.random(6000) < 0.4).astype(np.uint8)
        assert np.array_equal(dev.SetOccupancyBatchVox(vox, occ), ora.SetOccupancyBatchVox(vox, occ))
        assert dev.UpdateOccupancy(False) == ora.UpdateOccupancy(False)
        res = compare(dev, ora)
        assert res["occ"] == 0 and res["dist"] == 0 and res["cobs_tie"] == 0 and res["cobs_nontie"] == 0, ("after UpdateOccupancy", r, res)
        dev.UpdateESDF(); ora.UpdateESDF()
        res = compare(dev, ora)
        assert res["occ"] == 0 and res["dist"] == 0 and res["cobs_tie"] == 0 and res["cobs_nontie"] == 0, (r, res)
        assert dev.stats()["expansions"] == ora.stats()["expansions"], r
        D = ora.export_distance(); C = ora.export_closest_obstacle()
        seen_reset += int(((D == 10000) & (C[:, 0] != -10000)).sum())          # "distance infinity, obstacle kept" states persist
    assert seen_reset > 0
    q = rng.uniform(-2.5, 2.5, (256, 3)) * (1, 1, 0.5)
    d1, g1 = dev.GetDistWithGradTrilinearBatch(q); d2, g2 = ora.GetDistWithGradTrilinearBatch(q)
    assert np.array_equal(d1, d2) and np.array_equal(g1, g2)
    # the CUDA-graph query plan (fiesta_query_plan_*) returns the same bits, run after run
    plan = dev.QueryPlan(256)
    for rep in range(3):
        qq = q if rep == 0 else rng.uniform(-3.0, 3.0, (256, 3)) * (1, 1, 0.45)
        if rep == 2:
            qq[:8] = rng.uniform(4.0, 6.0, (8, 3))                # outside the map: -1 (ESDFMap.cpp:483-484), gradient untouched
        d3, g3 = plan.run(qq)
        d5, g5 = dev.GetDistWithGradTrilinearBatch(qq)            # the non-graph path: same kernel, same bits everywhere
        assert np.array_equal(d3, d5) and np.array_equal(g3, g5), rep
        d4, g4 = ora.GetDistWithGradTrilinearBatch(qq)
        ok = d4 != -1
        assert np.array_equal(d3, d4) and np.array_equal(g3[ok], g4[ok]), rep
    plan.close()


def test_device_resident_event_batch(oracle_built):
    """fiesta_set_occupancy_batch_vox_device == the host SetOccupancy loop (events already in HBM; dynamic-obstacle stress path)."""
    import torch
    dev, ora = pair(oracle_built, "fast", params=scenes.PARAMS_TOGGLE)
    allv = scenes.all_voxels(dev.grid_size)
    for m in (dev, ora):
        m.SetOccupancyBatchVox(allv, np.zeros(len(allv), np.uint8)); m.UpdateOccupancy(True); m.UpdateESDF()
    rng = np.random.default_rng(4)
    state = np.zeros(len(allv), np.uint8)
    for f in range(3):
        idx = rng.choice(len(allv), len(allv) // 5, replace=False)
        occ = (1 - state[idx]).astype(np.uint8); state[idx] = occ
        vox = np.concatenate([allv[idx], np.array([[-1, 0, 0], [10 ** 6, 2, 3]], np.int32)])   # + out-of-grid events: ignored
        occ2 = np.concatenate([occ, np.array([1, 1], np.uint8)])
        tv, to = torch.from_numpy(vox).cuda(), torch.from_numpy(occ2).cuda()
        dev.SetOccupancyBatchVoxDevice(tv.data_ptr(), to.data_ptr(), len(vox))
        ora.SetOccupancyBatchVox(allv[idx], occ)
        assert same_counters(dev, ora)
        assert dev.CheckUpdate() == ora.CheckUpdate()
        assert dev.UpdateOccupancy(True) == ora.UpdateOccupancy(True)
        dev.UpdateESDF(); ora.UpdateESDF()
        r = compare(dev, ora)
        # 20 % random occupancy is the regime where wave propagation (reference and FAST alike) is no longer an exact EDT and the
        # two make different choices at a handful of voxels; occupancy and counters stay identical
        assert r["occ"] == 0 and r["dist"] <= 1e-3 * r["finite"] and r["dist_max_err"] < 0.11, (f, r)


@pytest.mark.parametrize("mode,cap", [("exact", None), ("fast", None), ("exact", "64")])
def test_host_mirror_tracks_every_update(oracle_built, mode, cap, monkeypatch):
    """fiesta_host_mirror_* (SURVEY.md 8(f) #3): the pinned host records, patched with the changed entries after every update,
    answer GetDistance / GetDistWithGradTrilinear (ESDFMap.cpp:467-540) from host memory with the bits of the device queries --
    whole field and random positions, global and sliding local boxes, and through the bulk-copy path (change list of 64)."""
    if cap:
        monkeypatch.setenv("FIESTA_MIRROR_CAP", cap)
    dev, ora = pair(oracle_built, mode, params=scenes.PARAMS_TOGGLE)
    gs = dev.grid_size
    allv = scenes.all_voxels(gs)
    centres = (allv + 0.5) * 0.1 + np.array([-3.2, -3.2, -1.6])
    rng = np.random.default_rng(11)
    mir = dev.HostMirror()                                       # created on the empty map: everything unknown
    assert mir.refresh() == 0

    def check(tag):
        D = dev.export_distance()
        want = np.where(D < 0, 10000.0, D)                       # GetDistance reads unknown as +infinity_ (:478)
        assert np.array_equal(mir.GetDistanceBatch(centres), want), tag
        q = rng.uniform(-3.4, 3.4, (512, 3)) * (1, 1, 0.5)
        d1, g1 = dev.GetDistWithGradTrilinearBatch(q)
        d2, g2 = mir.GetDistWithGradTrilinearBatch(q)
        assert np.array_equal(d1, d2) and np.array_equal(g1, g2), tag
        assert np.array_equal(dev.GetDistanceBatch(q), mir.GetDistanceBatch(q)), tag
        if mode == "exact":                                      # and the reference's own answers where they are defined
            assert np.array_equal(mir.GetDistanceBatch(centres), ora.GetDistanceBatch(centres)), tag

    for m in (dev, ora):
        m.SetOccupancyBatchVox(allv, np.zeros(len(allv), np.uint8)); m.UpdateOccupancy(True); m.UpdateESDF()
    n = mir.refresh()
    assert n == len(allv) and mir.stats()["full_copies"] == (1 if cap else 0)
    check("observed")
    idx = rng.choice(len(allv), 200, replace=False)
    for m in (dev, ora):
        m.SetOccupancyBatchVox(allv[idx], np.ones(200, np.uint8)); m.UpdateOccupancy(True); m.UpdateESDF()
    assert mir.refresh() == len(allv)                            # every voxel got its first finite distance
    check("obstacles")
    for r in range(6):                                           # sliding local boxes, inserts and deletes
        c = np.array([-1.5 + 0.5 * r, -1.0 + 0.3 * r, 0.0])
        lo, hi = c - np.array([1.1, 1.0, 0.8]), c + np.array([1.1, 1.0, 0.8])
        vox = np.stack([rng.integers(0, gs[i], 3000) for i in range(3)], -1).astype(np.int32)
        occ = (rng.random(3000) < (1.0 if r < 3 else 0.4)).astype(np.uint8)       # rounds 0-2 only insert
        for m in (dev, ora):
            m.SetUpdateRange(lo, hi)
            m.SetOccupancyBatchVox(vox, occ); m.UpdateOccupancy(True); m.UpdateESDF()
        deletes = dev.stats()["deletes"]
        n = mir.refresh()
        st = mir.stats()
        assert st["changed"] == n and 0 < n < st["scanned"], (r, st)
        # inserts change records inside the update box only; a delete resets dependants anywhere (ESDFMap.cpp:301-334)
        assert (st["scanned"] == len(allv)) if deletes else (st["scanned"] < len(allv) // 2), (r, st, deletes)
        check(("box", r))
    assert mir.refresh() == 0 and mir.stats()["scanned"] == 0    # nothing happened since: nothing is scanned
    p = (0.31, -0.27, 0.12)
    assert mir.GetDistance(p) == dev.GetDistance(p)
    assert mir.GetDistance((10, 20, 5)) == dev.GetDistance((10, 20, 5))
    d1, g1 = mir.GetDistWithGradTrilinear(p); d2, g2 = dev.GetDistWithGradTrilinear(p)
    assert d1 == d2 and tuple(g1) == tuple(g2)
    assert mir.GetDistance((9.0, 0.0, 0.0)) == -10000 and mir.GetDistWithGradTrilinear((9.0, 0.0, 0.0))[0] == -1
    mir.close()


@pytest.mark.parametrize("mode", ["fast", "exact"])
def test_two_occupancy_updates_before_esdf(oracle_built, mode):
    """UpdateOccupancy twice, then one UpdateESDF: the insert / delete queues grow during the second call, and the pushes of the
    first one must survive that growth.  A grown queue holds 1.5x what was asked for plus 1 MiB (2^18 entries), so the second
    call pushes more than 2^18 crossings into each queue (EXACT), from every tile of the grid (FAST reserves 512 entries per
    touched tile).  The many voxels it deletes become occupied through a lowered threshold, not through inserts, so that the
    queues stay small until then."""
    origin = (-6.4, -6.4, -3.2)
    dev, ora = pair(oracle_built, mode, origin=origin, size=(12.8, 12.8, 6.4), params=scenes.PARAMS_DEFAULT)
    gs = dev.grid_size                                                       # 128 x 128 x 64: 2048 tiles
    allv = scenes.all_voxels(gs)
    slab = allv[allv[:, 0] < 40]                                             # 640 tiles
    rest = allv[allv[:, 0] >= 40]
    rng = np.random.default_rng(12)
    q = rest[rng.choice(np.flatnonzero(rest[:, 0] == 40), 50, replace=False)]
    fresh = rest[rest[:, 0] > 40]
    fresh = fresh[rng.permutation(len(fresh))]
    lowered = (0.70, 0.35, 0.12, 0.97, 0.60)                                 # one hit (0.847) is occupied, one more miss (0.228) is not

    def occupancy(vox, occ):
        assert np.array_equal(dev.SetOccupancyBatchVox(vox, occ), ora.SetOccupancyBatchVox(vox, occ))
        assert dev.UpdateOccupancy(True) == ora.UpdateOccupancy(True)

    occupancy(slab, np.ones(len(slab), np.uint8))                            # one hit each: below the default threshold
    for m in (dev, ora):
        m.SetParameters(*lowered)                                            # the whole slab is occupied now, no queue push
    occupancy(q, np.ones(len(q), np.uint8))                                  # 50 real obstacles next to the slab
    dev.UpdateESDF(); ora.UpdateESDF()
    occupancy(np.concatenate([q, fresh[:50]]), np.r_[np.zeros(50), np.ones(50)].astype(np.uint8))   # first call: 50 + 50
    big = fresh[50:270050]
    occupancy(np.concatenate([slab, big]), np.r_[np.zeros(len(slab)), np.ones(len(big))].astype(np.uint8))   # second call
    dev.UpdateESDF(); ora.UpdateESDF()
    sd, so = dev.stats(), ora.stats()
    assert (sd["inserts"], sd["deletes"]) == (so["inserts"], so["deletes"]) == (len(big) + 50, len(slab) + 50)
    if mode == "exact":
        r = compare(dev, ora)
        assert r["occ"] == 0 and r["dist"] == 0 and r["cobs_tie"] == 0 and r["cobs_nontie"] == 0, r
        assert sd["expansions"] == so["expansions"]
        pos = rng.uniform(-6.3, 6.2, (2000, 3)) * (1, 1, 0.5)
        d1, g1 = dev.GetDistWithGradTrilinearBatch(pos)
        d2, g2 = ora.GetDistWithGradTrilinearBatch(pos)
        assert np.array_equal(d1, d2) and np.array_equal(g1, g2)
    else:
        r = compare(dev, ora, check_counters=True)
        assert r["occ"] == 0 and r["counters"] == 0, r
        inv = invariants(dev, np.log(0.6 / 0.4))
        assert all(v == 0 for v in inv.values()), inv


def test_occupancy_threshold_change_exact(oracle_built):
    """SetParameters with a new p_occ on a map that already holds data (ESDFMap.cpp:218-224): Exist() (:46-48) follows the new
    threshold at once -- voxels between the two thresholds count as obstacles without ever having been inserted -- and every
    later delete / re-seeding decision uses it.  Arrays compared with the reference after every update."""
    dev, ora = pair(oracle_built, "exact")                                  # PARAMS_DEFAULT: two hits make a voxel occupied
    gs = dev.grid_size
    allv = scenes.all_voxels(gs)
    rng = np.random.default_rng(5)
    pick = rng.choice(len(allv), 900, replace=False)
    A, B = allv[pick[:500]], allv[pick[500:]]

    def step(vox, occ, tag):
        for m in (dev, ora):
            m.SetOccupancyBatchVox(vox, occ)
        assert dev.UpdateOccupancy(True) == ora.UpdateOccupancy(True), tag
        dev.UpdateESDF(); ora.UpdateESDF()
        res = compare(dev, ora)
        assert res["occ"] == 0 and res["dist"] == 0 and res["cobs_tie"] == 0 and res["cobs_nontie"] == 0, (tag, res)
        assert dev.stats()["expansions"] == ora.stats()["expansions"], tag

    step(allv, np.zeros(len(allv), np.uint8), "observe")
    step(np.concatenate([A, B]), np.ones(900, np.uint8), "hit 1")           # log-odds -0.619 + 0.847 = 0.228
    step(A, np.ones(500, np.uint8), "hit 2")                                # A 1.075: still below logit(0.8) = 1.386
    step(A, np.ones(500, np.uint8), "hit 3")                                # A 1.92: inserted.  B stays at 0.228 > logit(0.55) = 0.2
    assert dev.stats()["inserts"] == 500
    for m in (dev, ora):
        m.SetParameters(0.70, 0.35, 0.12, 0.97, 0.55)                       # B voxels now Exist() without an insert
    for r in range(5):
        n = 1200
        vox = np.concatenate([A[rng.choice(500, 150, replace=False)], B[rng.choice(400, 150, replace=False)],
                              np.stack([rng.integers(0, gs[i], n) for i in range(3)], -1).astype(np.int32)])
        occ = (rng.random(len(vox)) < 0.45).astype(np.uint8)
        step(vox, occ, ("after threshold change", r))
    for m in (dev, ora):
        m.SetParameters(*scenes.PARAMS_DEFAULT)                             # and back up
    for r in range(3):
        vox = np.stack([rng.integers(0, gs[i], 1500) for i in range(3)], -1).astype(np.int32)
        step(vox, (rng.random(1500) < 0.5).astype(np.uint8), ("threshold restored", r))
