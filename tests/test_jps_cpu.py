"""Host-side path search (fq_jps3d_plan*, faster_b200/csrc/fq_jps.cpp) against the REFERENCE's own graph search and planner
layer compiled from the original project (oracle/_ref/libjps_ref.so and libjpsplan_ref.so, built by oracle/Makefile with
stand-ins for boost::heap, Eigen, ROS and PCL).  What they returned on the inputs below is stored in
tests/golden/reference_jps.npz (tools/make_reference_goldens.py)."""
import functools
import os

import numpy as np
import pytest

from faster_b200 import capi

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_jps.npz")
RES, ORIGIN = 0.25, np.array([-5.0, -5.0, 0.0])


@functools.lru_cache(maxsize=None)
def reference(key):
    with np.load(GOLDEN) as z:
        return z[key]


def reference_paths(key):
    """The list of (n, 3) paths stored under `key` (rows of all paths, and each path's length)."""
    pts, n = reference(key + ".points"), reference(key + ".n")
    ends = np.cumsum(n)
    return [pts[e - k:e] for k, e in zip(n, ends)]


def _forest_grid(seed, dims=(40, 40, 12), res=0.25, n_trees=28):
    rng = np.random.default_rng(seed)
    xd, yd, zd = dims
    g = np.zeros((zd, yd, xd), np.int8)
    for _ in range(n_trees):
        cx, cy = rng.uniform(0, xd * res), rng.uniform(0, yd * res)
        r = rng.uniform(0.15, 0.6)
        xs, ys = np.meshgrid((np.arange(xd) + 0.5) * res, (np.arange(yd) + 0.5) * res)
        g[:, ((xs - cx) ** 2 + (ys - cy) ** 2 <= r * r)] = 100
    for _ in range(6):                                   # a few floating boxes and unknown pockets
        x0, y0, z0 = rng.integers(0, xd - 6), rng.integers(0, yd - 6), rng.integers(0, zd - 3)
        g[z0:z0 + rng.integers(1, 4), y0:y0 + rng.integers(2, 7), x0:x0 + rng.integers(2, 7)] = 100 if rng.uniform() < 0.7 else -1
    return g


def _free_cell(g, rng):
    zd, yd, xd = g.shape
    for _ in range(1000):
        c = (int(rng.integers(0, xd)), int(rng.integers(0, yd)), int(rng.integers(0, zd)))
        if g[c[2], c[1], c[0]] == 0:
            return c
    raise RuntimeError


def _check_path(g, path, cost):
    """consecutive points are joined by straight runs along one of the 26 directions through free cells."""
    total = 0.0
    for a, b in zip(path[:-1], path[1:]):
        d = b - a
        n = np.abs(d).max()
        assert n > 0 and np.all((np.abs(d) == n) | (d == 0)), "not a 26-direction run"
        step = d // n
        for k in range(1, n + 1):
            c = a + k * step
            assert g[c[2], c[1], c[0]] == 0
        total += n * np.sqrt(float(np.sum(step * step)))
    assert abs(total - cost) <= 1e-9 * max(1.0, cost)


def map_queries(seed):
    """The random map of test_costs_equal_the_reference_on_random_maps and its 12 (start, goal) pairs."""
    g = _forest_grid(seed)
    rng = np.random.default_rng(100 + seed)
    return g, [(_free_cell(g, rng), _free_cell(g, rng)) for _ in range(12)]


def hole_map():
    """A wall splits the map; one hole in it."""
    g = np.zeros((6, 12, 12), np.int8)
    g[:, :, 6] = 100
    g[2, 5, 6] = 0
    return g


def world_queries():
    """(grid, world start, world goal) of test_world_plan_equals_the_reference_planner: 40 forest maps, then the refusals (an
    occupied start, an occupied goal, a walled-in goal)."""
    out = []
    for seed in range(40):
        g = _forest_grid(50 + seed)
        rng = np.random.default_rng(seed)
        s, t = _free_cell(g, rng), _free_cell(g, rng)
        ws = (np.array(s) + 0.5) * RES + ORIGIN + rng.uniform(-0.1, 0.1, 3)
        wt = (np.array(t) + 0.5) * RES + ORIGIN + rng.uniform(-0.1, 0.1, 3)
        out.append((g, ws, wt))
    g = _forest_grid(7)
    occ = np.argwhere(g == 100)[0][::-1]
    free = np.array(_free_cell(g, np.random.default_rng(1)))
    w_occ, w_free = (occ + 0.5) * RES + ORIGIN, (free + 0.5) * RES + ORIGIN
    out += [(g, w_occ, w_free), (g, w_free, w_occ)]
    g2 = np.zeros((6, 12, 12), np.int8)
    g2[:, 4:9, 4] = g2[:, 4:9, 8] = g2[:, 4, 4:9] = g2[:, 8, 4:9] = 100
    g2[0, 4:9, 4:9] = g2[5, 4:9, 4:9] = 100                          # a closed box around the goal
    out.append((g2, (np.array([1, 1, 2]) + 0.5) * RES + ORIGIN, (np.array([6, 6, 2]) + 0.5) * RES + ORIGIN))
    return out


def test_pruning_rules_equal_the_reference_tables(built_lib):
    ns, f1, f2, cnt = capi.jps3d_rules()
    rn, rf1, rf2 = reference("tables.ns"), reference("tables.f1"), reference("tables.f2")
    nsz = {0: (26, 0), 1: (1, 8), 2: (3, 12), 3: (7, 12)}          # graph_search.h:123-135
    distinct = {1: 8, 2: 8, 3: 6}                                     # blockers hasForced() looks at (:420-470)
    for dz in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                i = (dx + 1) + 3 * (dy + 1) + 9 * (dz + 1)
                n1 = abs(dx) + abs(dy) + abs(dz)
                a, b = nsz[n1]
                assert tuple(cnt[i]) == (a, b)
                assert {tuple(ns[i, :, k]) for k in range(a)} == {tuple(rn[i, :, k]) for k in range(a)}
                mine = sorted((tuple(f1[i, :, k]), tuple(f2[i, :, k])) for k in range(b))
                ref = sorted((tuple(rf1[i, :, k]), tuple(rf2[i, :, k])) for k in range(b))
                assert mine == ref
                if n1:
                    assert {tuple(f1[i, :, k]) for k in range(b)} == {tuple(rf1[i, :, k]) for k in range(distinct[n1])}


@pytest.mark.parametrize("seed", range(8))
def test_costs_equal_the_reference_on_random_maps(built_lib, seed):
    g, queries = map_queries(seed)
    ref = reference("maps")[seed]                          # per query: JPS found, JPS cost, A* found, A* cost
    solved = 0
    for (s, t), (rj, rcj, ra, rca) in zip(queries, ref):
        pj, cj, ej = capi.jps3d_plan(g, s, t, True)
        pa, ca, ea = capi.jps3d_plan(g, s, t, False)
        assert (len(pj) > 0) == (len(pa) > 0)
        assert bool(rj) == (len(pj) > 0) and bool(ra) == (len(pa) > 0)
        if len(pj) == 0:
            continue
        solved += 1
        assert abs(cj - ca) <= 1e-9 * ca, "JPS and A* disagree"
        assert tuple(pj[0]) == s and tuple(pj[-1]) == t and tuple(pa[0]) == s and tuple(pa[-1]) == t
        _check_path(g, pj, cj)
        _check_path(g, pa, ca)
        assert ej <= ea                                   # jump points: never more expansions than A*
        assert abs(cj - rcj) <= 1e-9 * rcj and abs(ca - rca) <= 1e-9 * rca
    assert solved >= 6


def test_unreachable_blocked_and_trivial(built_lib):
    g = np.zeros((6, 12, 12), np.int8)
    g[:, :, 6] = 100                                      # a wall splits the map
    p, c, _ = capi.jps3d_plan(g, (1, 1, 1), (10, 10, 4), True)
    assert len(p) == 0 and np.isinf(c)
    g = hole_map()
    p, c, _ = capi.jps3d_plan(g, (1, 1, 1), (10, 10, 4), True)
    pa, ca, _ = capi.jps3d_plan(g, (1, 1, 1), (10, 10, 4), False)
    assert len(p) > 0 and abs(c - ca) < 1e-9 and any(tuple(q) == (6, 5, 2) for q in pa)
    assert abs(reference("hole_cost") - c) < 1e-9
    assert len(capi.jps3d_plan(g, (6, 0, 0), (1, 1, 1), True)[0]) == 0          # start occupied
    assert len(capi.jps3d_plan(g, (1, 1, 1), (40, 1, 1), True)[0]) == 0         # goal outside
    p, c, _ = capi.jps3d_plan(g, (3, 3, 3), (3, 3, 3), True)                    # start == goal
    assert len(p) == 1 and c == 0.0
    g[:] = -1                                             # unknown cells cannot be entered
    g[1, 1, 1] = 0
    g[1, 1, 2] = 0
    assert capi.jps3d_plan(g, (1, 1, 1), (2, 1, 1), True)[1] == 1.0


def test_world_plan_post_processing(built_lib):
    """fq_jps3d_plan_world: cell centres (map_util.h:334-347), line points removed, corners cut while the straight line
    stays clear of occupied cells (jps_planner.cpp:36-105)."""
    res, origin = 0.25, np.array([-5.0, -5.0, 0.0])
    n_ok = 0
    for seed in range(6):
        g = _forest_grid(50 + seed)
        rng = np.random.default_rng(seed)
        s, t = _free_cell(g, rng), _free_cell(g, rng)
        ws = (np.array(s) + 0.5) * res + origin + rng.uniform(-0.1, 0.1, 3)
        wt = (np.array(t) + 0.5) * res + origin
        path, raw = capi.jps3d_plan_world(g, origin, res, ws, wt, True)
        cells, c, _ = capi.jps3d_plan(g, s, t, True)
        if len(cells) == 0:
            assert len(path) == 0
            continue
        n_ok += 1
        assert abs(raw - c * res) <= 1e-9
        assert np.allclose(path[0], (np.array(s) + 0.5) * res + origin) and np.allclose(path[-1], (np.array(t) + 0.5) * res + origin)
        length = np.sum(np.linalg.norm(np.diff(path, axis=0), axis=1))
        assert length <= raw + 1e-9 and len(path) <= len(cells)
        for a, b in zip(path[:-1], path[1:]):            # every kept segment has line of sight (ray traced at 0.8 cell)
            m = int(np.abs((b - a) / res).max() / 0.8)
            for k in range(1, m):
                pt = a + (b - a) * (k / m)
                cidx = np.round((pt - origin) / res - 0.5).astype(int)
                assert g[cidx[2], cidx[1], cidx[0]] < 100
    assert n_ok >= 3


def test_world_plan_equals_the_reference_planner(built_lib):
    """fq_jps3d_plan_world against the REFERENCE's own planner layer compiled from the original project (JPSPlanner<3>::plan over
    MapUtil<3>: floatToInt / intToFloat, graph search, removeLinePts, removeCornerPts forwards and backwards with the
    ray-traced line of sight -- jps_planner.cpp:196-295, map_util.h:334-383): the same way points, bit for bit, with JPS and
    with plain A*; the same refusals (start or goal not free, no path)."""
    res, origin = RES, ORIGIN
    queries = world_queries()
    refs = list(zip(reference_paths("world.path"), reference_paths("world.raw"), reference("world.status")))
    assert len(refs) == 2 * len(queries)                  # JPS, then A*, per query
    n_paths = n_simplified = 0
    for seed, (g, ws, wt) in enumerate(queries[:40]):
        for k, use_jps in enumerate((True, False)):
            ours, raw_len = capi.jps3d_plan_world(g, origin, res, ws, wt, use_jps)
            ref, raw, status = refs[2 * seed + k]
            assert len(ours) == len(ref), (seed, use_jps, status)
            if len(ref):
                assert np.array_equal(ours, ref), (seed, use_jps, np.abs(ours - ref).max())
                assert abs(raw_len - np.sum(np.linalg.norm(np.diff(raw, axis=0), axis=1))) <= 1e-9
                n_paths += 1
                n_simplified += len(ref) < len(raw)
    assert n_paths >= 60 and n_simplified >= 40
    # refusals: an occupied start, an occupied goal, a walled-in goal (JPS)
    for q, (g, a, b) in enumerate(queries[40:]):
        ours, _ = capi.jps3d_plan_world(g, origin, res, a, b, True)
        ref, _, status = refs[2 * (40 + q)]
        assert len(ours) == 0 and len(ref) == 0 and status in ((1, 2) if q < 2 else (-1,))
