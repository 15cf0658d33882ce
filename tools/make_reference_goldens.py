#!/usr/bin/env python
"""Golden outputs of THE REFERENCE ITSELF for the tests that compare with it: its solverGurobi.cpp, DecompUtil and JPS3D code
compiled unmodified into oracle/_ref/ by oracle/Makefile (needs the original project's tree: make -C oracle REFROOT=...), run on
the inputs those tests generate (their own input functions are imported, so both sides see the same numbers).  Writes
  tests/golden/reference_solver.npz  -- tests/test_reference_solver_cpu.py: the model of one trial, getDTInitial, fillX, and
                                        genNewTraj's loop with HiGHS + enumeration of the binaries answering optimize();
  tests/golden/reference_decomp.npz  -- tests/test_decomp_cpu.py: the polytopes of EllipsoidDecomp3D;
  tests/golden/reference_jps.npz     -- tests/test_jps_cpu.py: pruning tables, graph-search costs, planner way points.
The tests then run wherever the repository is checked out, without the original project."""
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from faster_b200 import capi                                                   # noqa: E402
from oracle import decomp_ref as dref, jps_ref, model_fullspace as mf, solver_ref as sr      # noqa: E402
import test_decomp_cpu as td                                                   # noqa: E402
import test_jps_cpu as tj                                                      # noqa: E402
import test_reference_solver_cpu as ts                                         # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def highs(q, Aeq, beq, Ain, bin_):
    ok, z = mf.solve_qp_highs(sp.diags(2.0 * q).tocsc(), Aeq, beq, Ain, bin_)
    return ok, z, (float(np.sum(q * z * z)) if ok else np.inf)


def loop_result(r):
    """genNewTraj's result with every 16th sampled state and the last one (fillX itself is compared in full on its own)."""
    s = r.pop("samples")
    rows = np.unique(np.r_[np.arange(0, len(s), 16), len(s) - 1]) if len(s) else np.zeros(0, np.int64)
    return dict(r, n_samples=len(s), sample_rows=rows, samples=s[rows])


def put(out, key, d):
    for k, v in d.items():
        out[key + "." + k] = np.asarray(v)


def solver_goldens():
    out = {}
    for name, N, P, ff, profile in ts.CASES:
        pb, polys = ts.model_corridor(N, P, ff, profile)
        base = max(capi.dt_initial(pb["x0"], pb["xf"], pb["lim"], N), 0.02)
        for k, dt in enumerate((1.3 * base, 2.7 * base)):
            md = sr.model(N, pb["x0"], pb["xf"], pb["lim"], dt, polys, ff)
            A = sp.csr_matrix(md.pop("A"))
            assert A.shape[1] < 2 ** 15 and np.diff(A.indptr).max() < 2 ** 8
            put(out, "model.%s.%d" % (name, k), dict(md, dt=dt, A_shape=A.shape, A_row_nnz=np.diff(A.indptr).astype(np.uint8),
                                                      A_indices=A.indices.astype(np.int16), A_vals=A.data))
    inputs, edge = ts.dt_initial_inputs()
    out["dt_initial"] = np.array([sr.dt_initial(*a) for a in inputs])
    out["dt_initial_edge"] = np.array([sr.dt_initial(*a) for a in edge])
    for seed, (N, dt, DC) in enumerate(ts.FILL_X_CASES):
        out["fill_x.%d" % seed] = sr.fill_x(N, np.random.default_rng(seed).normal(size=(N, 12)), dt, DC)
    for N, P, ff in ts.LOOP_CASES:
        for seed in range(3):
            pb, polys = ts.loop_corridor(N, P, ff, seed)
            put(out, "loop.%d.%d.%d.%d" % (N, P, ff, seed),
                loop_result(sr.gen_new_traj(N, pb["x0"], pb["xf"], pb["lim"], polys, 0.01, 1.0, 6.0, 1.0, highs, ff)))
    pb, far = ts.refusal_corridor()
    put(out, "refusal.far", loop_result(sr.gen_new_traj(4, pb["x0"], far, pb["lim"], pb["polys"], 0.01, 1.0, 3.0, 1.0, highs, True)))
    stopped = sr.gen_new_traj(4, pb["x0"], pb["xf"], pb["lim"], pb["polys"], 0.01, 1.0, 3.0, 1.0, highs, True, stop_first=True)
    put(out, "refusal.stopped", {k: stopped[k] for k in ("solved", "trials", "n_optimize")})     # no trial ran: dt_ is never set
    return out


def put_polys(out, key, calls):
    """Lists of polytopes (one list per call) -> all rows, rows per polytope, polytopes per call."""
    flat = [np.hstack([A, b[:, None]]) for polys in calls for A, b in polys]
    out[key + ".Ab"] = np.vstack(flat)
    out[key + ".rows"] = np.array([len(x) for x in flat], np.int32)
    out[key + ".polys"] = np.array([len(polys) for polys in calls], np.int32)


def decomp_goldens():
    out = {}
    put_polys(out, "product", [dref.cvx_ellipsoid_decomp(p, o, (2.0, 2.0, 1.0), r, 0.0) for p, o, r in td._clouds(1, 45)])
    put_polys(out, "restatement", [dref.cvx_ellipsoid_decomp(p, o, (2.0, 2.0, 1.0), r, 0.0) for p, o, r in td._clouds(2, 30)])
    put_polys(out, "demo", [dref.cvx_ellipsoid_decomp(td.DEMO_PATH, np.zeros((0, 3)), (1.0, 2.0, 1.0), 0.0, -100.0)])
    put_polys(out, "edge", [dref.cvx_ellipsoid_decomp(p, o, inflate=r) for p, o, r in td.EDGE_CASES])
    return out


def put_paths(out, key, paths):
    out[key + ".points"] = np.vstack([np.reshape(p, (-1, 3)) for p in paths])
    out[key + ".n"] = np.array([len(p) for p in paths], np.int32)


def jps_goldens():
    assert jps_ref.available() and jps_ref.planner_available()
    out = {}
    ns, f1, f2 = jps_ref.tables()
    n1 = np.abs(np.indices((3, 3, 3)) - 1).sum(axis=0).reshape(27)        # nonzero components of direction (dx, dy, dz)
    for table, count in ((ns, np.array([26, 1, 3, 7])[n1]), (f1, np.array([0, 8, 12, 12])[n1]), (f2, np.array([0, 8, 12, 12])[n1])):
        table[np.arange(table.shape[2])[None, None, :] >= count[:, None, None]] = 0          # slots past the counts are never written
    out["tables.ns"], out["tables.f1"], out["tables.f2"] = ns, f1, f2
    maps = np.zeros((8, 12, 4))
    for seed in range(8):
        g, queries = tj.map_queries(seed)
        for q, (s, t) in enumerate(queries):
            rj, rcj, _ = jps_ref.plan(g, s, t, True)
            ra, rca, _ = jps_ref.plan(g, s, t, False)
            maps[seed, q] = (len(rj) > 0, rcj, len(ra) > 0, rca)
    out["maps"] = maps
    out["hole_cost"] = np.float64(jps_ref.plan(tj.hole_map(), (1, 1, 1), (10, 10, 4), True)[1])
    paths, raws, status = [], [], []
    for g, ws, wt in tj.world_queries():
        for use_jps in (True, False):
            p, raw, st = jps_ref.plan_world(g, tj.ORIGIN, tj.RES, ws, wt, use_jps)
            paths.append(p); raws.append(raw); status.append(st)
    put_paths(out, "world.path", paths)
    put_paths(out, "world.raw", raws)
    out["world.status"] = np.array(status, np.int32)
    return out


if __name__ == "__main__":
    assert sr.available() and dref.available(), "build oracle/_ref first: make -C oracle REFROOT=<the original project>"
    for name, make in (("reference_solver.npz", solver_goldens), ("reference_decomp.npz", decomp_goldens),
                       ("reference_jps.npz", jps_goldens)):
        path = os.path.join(GOLDEN, name)
        np.savez_compressed(path, **make())
        print("wrote", path, os.path.getsize(path), "bytes")
