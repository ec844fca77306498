"""Generates tests/golden/*.json by running the UNMODIFIED reference (oracle/_ref/libfiesta_ref.so, compiled in place from
/root/reference by oracle/Makefile).  Run in the dev container (the only place /root/reference exists):

    python tests/golden/make_golden.py

The JSON files pin the C restatement (oracle/esdf_oracle.c) and the CUDA path on machines without the reference.
Array-valued results are stored as SHA-256 digests plus a few sampled values.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle  # noqa: E402
from tests import scenes  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def checkpoint(m):
    D = m.export_distance()
    O = m.export_occupancy()
    fin = (D >= 0) & (D < 10000)
    st = m.stats()
    return dict(occupied=int((O > np.log(0.8 / 0.2)).sum()), finite=int(fin.sum()), sum_distance=float(D[fin].sum()),
                accumulator=int(st["accumulator"]), expansions=int(st["expansions"]), change_num=int(st["change_num"]),
                consistent=bool(m.CheckConsistency()), distance_sha256=digest(D), occupancy_sha256=digest(O),
                closest_obstacle_sha256=digest(m.export_closest_obstacle()))


def step(m, vox, occ):
    m.SetOccupancyBatchVox(vox, occ)
    m.UpdateOccupancy(True)
    m.UpdateESDF()


def pillar_replay(kind):
    """SURVEY.md 8(d) config 1 / Appendix D."""
    m = pyoracle.OracleMap((-6.4, -6.4, 0.0), 0.2, (12.8, 12.8, 12.8), kind)
    m.SetParameters(*scenes.PARAMS_TOGGLE)
    out = {}
    allv = scenes.all_voxels(m.grid_size)
    step(m, allv, np.zeros(len(allv), np.uint8))
    out["after_observe_all"] = checkpoint(m)
    sites = scenes.pillar_sites()
    for k, (x, y) in enumerate(sites):
        step(m, scenes.pillar(x, y), np.ones(25, np.uint8))
        if k in (0, 24):
            out["after_pillar_%d" % k] = checkpoint(m)
    out["GetDistance_30_30_10"] = m.GetDistance((30, 30, 10))
    d, g = m.GetDistWithGradTrilinear((0.33, -1.27, 2.51))
    out["trilinear_0.33_-1.27_2.51"] = dict(dist=d, grad=list(map(float, g)))
    for k, (x, y) in enumerate(reversed(sites)):
        step(m, scenes.pillar(x, y), np.zeros(25, np.uint8))
        if k in (12, 24):
            out["after_delete_%d" % k] = checkpoint(m)
    return out


def random_replay(kind):
    """Partially observed 40^3 grid, 6 rounds of mixed SetOccupancy events (seed 11)."""
    rng = np.random.default_rng(11)
    m = pyoracle.OracleMap((-2.0, -2.0, -2.0), 0.1, (4.0, 4.0, 4.0), kind)
    m.SetParameters(*scenes.PARAMS_TOGGLE)
    out = {"grid_size": list(m.grid_size), "rounds": []}
    for r in range(6):
        n = 20000 if r == 0 else 3000
        vox = np.stack([rng.integers(0, m.grid_size[i], n) for i in range(3)], -1).astype(np.int32)
        occ = (rng.random(n) < (0.02 if r == 0 else 0.4)).astype(np.uint8)
        idx = m.SetOccupancyBatchVox(vox, occ)
        m.UpdateOccupancy(True)
        m.UpdateESDF()
        c = checkpoint(m)
        c["set_occupancy_returns_sha256"] = digest(idx)
        out["rounds"].append(c)
    pos = rng.uniform(-1.9, 1.9, (64, 3))
    d, g = m.GetDistWithGradTrilinearBatch(pos)
    out["query_positions"] = pos.tolist()
    out["query_dist"] = d.tolist()
    out["query_grad"] = g.tolist()
    return out


def raycast_replay(kind):
    """3 reduced-resolution depth frames into a 128x128x64 grid at 0.1 m, default probabilities (seed 2/3)."""
    m = pyoracle.OracleMap((-6.4, -6.4, -3.2), 0.1, (12.8, 12.8, 6.4), kind)
    m.SetParameters(*scenes.PARAMS_DEFAULT)
    sc = scenes.Scene((5.0, 5.0, 2.5), 20, 5, seed=2)
    out = {"frames": []}
    for p, yaw in scenes.pose_walk(3, seed=3):
        pts, T = scenes.depth_frame(sc, p, yaw, width=160, height=120, scale=0.25)
        cast = m.RaycastFrame(pts, T, 0.5, 5.0)
        hit, tot = m.export_counters()
        fr = dict(points_sha256=digest(pts), rays_cast=int(cast), touched=int((tot > 0).sum()), sum_hit=int(hit.sum()),
                  sum_total=int(tot.sum()), hit_sha256=digest(hit), total_sha256=digest(tot))
        m.UpdateOccupancy(True)
        m.UpdateESDF()
        fr.update(checkpoint(m))
        out["frames"].append(fr)
        sc.step()
    return out


def mixed_replay(kind):
    """32^3 grid, 5 rounds of 5000 SetOccupancy events (seed 5), a local update box in round 3, then batch queries and the
    sentinel returns (ESDFMap.cpp:402-410)."""
    rng = np.random.default_rng(5)
    m = pyoracle.OracleMap((-1.6, -1.6, -1.6), 0.1, (3.15, 3.15, 3.15), kind)
    m.SetParameters(*scenes.PARAMS_TOGGLE)
    out = {"grid_size": list(m.grid_size), "rounds": []}
    for r in range(5):
        n = 5000
        vox = rng.integers(0, m.grid_size[0], (n, 3)).astype(np.int32)
        occ = (rng.random(n) < 0.1).astype(np.uint8)
        idx = m.SetOccupancyBatchVox(vox, occ)
        if r == 3:   # local update box
            m.SetUpdateRange((-1.0, -1.0, -1.0), (1.0, 0.8, 0.6))
        changed = m.UpdateOccupancy(r != 3)
        m.UpdateESDF()
        c = checkpoint(m)
        c.update(set_occupancy_returns_sha256=digest(idx), update_occupancy=bool(changed), stats=m.stats())
        out["rounds"].append(c)
        if r == 3:
            m.SetOriginalRange()
    pos = rng.uniform(-1.8, 1.8, (3000, 3))
    d, g = m.GetDistWithGradTrilinearBatch(pos * 0.8)
    out.update(distance_batch_sha256=digest(m.GetDistanceBatch(pos)), trilinear_dist_sha256=digest(d), trilinear_grad_sha256=digest(g),
               sentinel_set_occupancy_bad_value=m.SetOccupancy((0.0, 0.0, 0.0), 2),
               sentinel_set_occupancy_out_of_map=m.SetOccupancy((9.0, 0.0, 0.0), 1),
               sentinel_get_distance_out_of_map=m.GetDistance((9.0, 0.0, 0.0)),
               sentinel_trilinear_out_of_map=m.GetDistWithGradTrilinear((9.0, 0.0, 0.0))[0])
    return out


VIS_MAP = ((-3.2, -3.2, -1.6), 0.1, (6.4, 6.4, 3.2))


def vis_replay(m):
    """GetPointCloud / GetSliceMarker of map `m` (built with VIS_MAP) after 4 depth frames (seed 5/6), then inside a local
    visualisation box (Fiesta.h:150).  Takes the map so the GPU test can drive the CUDA path through the same sequence."""
    m.SetParameters(*scenes.PARAMS_DEFAULT)
    sc = scenes.Scene((2.8, 2.8, 1.4), 8, 2, seed=5, edge=(0.3, 0.8))
    for p, yaw in scenes.pose_walk(4, seed=6, clamp=0.5):
        pts, T = scenes.depth_frame(sc, p, yaw, width=160, height=120, scale=0.25)
        m.RaycastFrame(pts, T, 0.3, 4.0)
        m.UpdateOccupancy(True)
        m.UpdateESDF()
        sc.step()

    def cloud(lo, hi):
        a = m.GetPointCloud(lo, hi)
        return dict(n=len(a), sha256=digest(a))

    def marker(sl, max_dist):
        xyz, rgba = m.GetSliceMarker(sl, max_dist)
        return dict(n=len(xyz), xyz_sha256=digest(xyz), rgba_sha256=digest(rgba))

    out = {"point_cloud_0_31": cloud(0, 31), "point_cloud_10_20": cloud(10, 20)}
    for sl in (0, 12, 16, 31):
        out["slice_%d_2.0" % sl] = marker(sl, 2.0)
    m.SetUpdateRange((-1.0, -1.5, -0.5), (2.0, 1.0, 0.7), False)
    out["local_point_cloud_0_31"] = cloud(0, 31)
    out["local_slice_14_1.0"] = marker(14, 1.0)
    return out


def dda_vectors(kind):
    """Raycast() known answers, including SURVEY.md Appendix B cases."""
    cases = [((1.5, 1.5, 1.5), (6.2, 3.7, 1.9)), ((6.2, 3.7, 1.9), (1.5, 1.5, 1.5)), ((2.0, 2.0, 2.0), (5.0, 5.0, 5.0)),
             ((1.2, 1.3, 1.4), (1.7, 1.8, 1.9)), ((-3.5, 2.5, 0.5), (12.25, -7.75, 3.125)), ((20.5, 20.5, 20.5), (2.5, 3.5, 4.5))]
    out = []
    for s, e in cases:
        r = pyoracle.raycast(s, e, (0, 0, 0), (16, 16, 16), kind)
        out.append(dict(start=s, end=e, min=(0, 0, 0), max=(16, 16, 16), voxels=r.tolist()))
    return out


if __name__ == "__main__":
    assert pyoracle.available("ref"), "oracle/_ref is not built: run `make -C oracle ref` where /root/reference exists"
    gold = dict(generator="tests/golden/make_golden.py", source="oracle/_ref (unmodified reference ESDFMap.cpp + raycast.cpp)",
                pillar_replay=pillar_replay("ref"), random_replay=random_replay("ref"), raycast_replay=raycast_replay("ref"),
                dda=dda_vectors("ref"), mixed_replay=mixed_replay("ref"),
                vis_replay=vis_replay(pyoracle.OracleMap(*VIS_MAP, kind="ref")))
    with open(os.path.join(HERE, "reference_golden.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
    print("wrote", os.path.join(HERE, "reference_golden.json"))
