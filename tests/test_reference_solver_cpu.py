"""The hot path against THE REFERENCE'S OWN CODE: faster/src/solverGurobi.cpp compiled unmodified from the original project
(oracle/Makefile -> oracle/_ref/libsolver_ref.so) over a recording stand-in for the Gurobi C++ API (oracle/stub_gurobi) and a
minimal Eigen stand-in (oracle/stub_eigen).  Gurobi's numerical solve is the one thing that cannot run here (closed source);
everything the reference does around it does.  What that compiled code returned on the inputs below is stored in
tests/golden/reference_solver.npz (tools/make_reference_goldens.py), so these comparisons run on every checkout:

  * the MODEL -- variables, cost, initial / final / continuity rows, box rows, binaries and indicator rows over the Bezier
    control points -- is read back from the reference's own model-building functions and compared, row by row, with the
    literal restatement every other parity test of this repository rests on (oracle/model_fullspace.build);
  * getDTInitial, resetX and fillX are compared with the product's host functions (fq_dt_initial, fq_num_samples, fq_fill_x);
  * genNewTraj's factor loop runs end to end with an independent solver (HiGHS + enumeration of the binaries) answering
    optimize(), and is compared with the sweep of the CPU restatement (oracle/fq_oracle.c), which the GPU tests compare the
    CUDA path with.
"""
import functools
import os

import numpy as np
import pytest
import scipy.sparse as sp

from faster_b200 import capi, corridor as cr
from oracle import model_fullspace as mf, solver_ref as sr

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_solver.npz")

CASES = [("cfg1", 3, 0, True, "uav"), ("cfg2", 10, 3, True, "uav"), ("cfg3", 10, 4, False, "uav"), ("cfg5", 15, 8, True, "ground"),
         ("yaml", 6, 3, True, "uav"), ("safe-small", 6, 2, False, "uav")]
LOOP_CASES = [(5, 2, True), (4, 3, True), (5, 2, False), (4, 0, True)]
FILL_X_CASES = [(10, 0.37, 0.01), (6, 0.2051, 0.01), (15, 0.113, 0.01), (3, 0.5, 0.05), (10, 0.0012, 0.01)]


@functools.lru_cache(maxsize=None)
def _golden():
    with np.load(GOLDEN) as z:
        return dict(z)


def reference(key):
    """The reference's output stored under `key` (tools/make_reference_goldens.py): an array, or a dict of its fields."""
    g = _golden()
    if key in g:
        return g[key]
    d = {k[len(key) + 1:]: v for k, v in g.items() if k.startswith(key + ".")}
    assert d, "no golden entry %r" % key
    return {k: (v[()] if v.ndim == 0 else v) for k, v in d.items()}


def reference_model(name, k):
    """The model of reference(...) with its sparse matrix made dense again: the layout of oracle.solver_ref.model."""
    md = reference("model.%s.%d" % (name, k))
    indptr = np.concatenate([[0], np.cumsum(md.pop("A_row_nnz"), dtype=np.int64)])
    A = sp.csr_matrix((md.pop("A_vals"), md.pop("A_indices").astype(np.int64), indptr), shape=tuple(md.pop("A_shape")))
    return dict(md, A=A.toarray())


def model_corridor(N, P, ff, profile):
    pb = cr.make_corridor(7000 + N + P, max(P, 1), N, profile, ff)
    return pb, (pb["polys"] if P else [])


def dt_initial_inputs():
    """400 random (x0, xf, lim, N), then edge cases."""
    rng = np.random.default_rng(3)
    out = []
    for k in range(400):
        x0 = np.concatenate([rng.uniform(-5, 5, 3), rng.uniform(-3, 3, 3), rng.uniform(-2, 2, 3)])
        xf = np.concatenate([x0[:3] + rng.uniform(-6, 6, 3), rng.uniform(-1, 1, 3) * (k % 2), np.zeros(3)])
        if k % 7 == 0:
            xf[1:3] = x0[1:3]                                    # axes without displacement
        lim = [[5, 5, 8], [1.4, 1.4, 5.0], [2, 3, 10]][k % 3]
        N = [3, 6, 10, 15][k % 4]
        out.append((x0, xf, lim, N))
    z = np.zeros(9)
    edge = [(z, z, [5, 5, 8], 10)]                                # identical rest states: 0 (findDT then takes 2 DC)
    far = z.copy(); far[0] = 1e6
    edge.append((z, far, [5, 5, 8], 10))                          # "no solution" branch: > 10000 s -> 0 (:752-756)
    nm = z.copy(); nm[:3] = [1e-9, -1e-9, 0.0]
    edge.append((z, nm, [5, 5, 8], 10))
    fast = z.copy(); fast[3:6] = [4.9, -4.9, 0.0]
    near = z.copy(); near[:3] = [0.5, -0.5, 0.1]
    edge.append((fast, near, [5, 5, 8], 6))
    acc = z.copy(); acc[6:9] = [2.9, -2.9, 1.0]
    back = z.copy(); back[:3] = [-3, 3, 1]
    edge.append((acc, back, [5, 3, 5], 10))
    away = z.copy(); away[3] = 1.0
    goal = z.copy(); goal[0] = -2.0
    edge.append((away, goal, [1.4, 1.4, 5.0], 15))
    return out, edge


def loop_corridor(N, P, ff, seed):
    pb = cr.make_corridor(910 + 10 * N + seed, max(P, 1), N, "uav", ff)
    return pb, (pb["polys"] if P else [])


def refusal_corridor():
    pb = cr.make_corridor(955, 2, 4, "uav", True)
    far = np.array(pb["xf"], float)
    far[:3] += 40.0                                              # a goal far outside the corridor
    return pb, far


@pytest.mark.parametrize("name,N,P,ff,profile", CASES)
def test_literal_model_equals_what_the_reference_code_builds(name, N, P, ff, profile):
    """oracle/model_fullspace.build against the rows the reference's createVars / setBounds / setPolytopesConstraints /
    setConstraintsX0 / setConstraintsXf / setDynamicConstraints / setObjective create (solverGurobi.cpp:70-120,:180-291,
    :332-407,:499-524): EXACTLY equal coefficients and right-hand sides (the same arithmetic on the same numbers); equalities and
    box rows in the same order, the corridor rows of a segment grouped by face then control point in the reference and by control
    point then face in the restatement.  The two time allocations are 1.3 and 2.7 times getDTInitial's value."""
    rng = np.random.default_rng(len(name) + N)
    pb, polys = model_corridor(N, P, ff, profile)
    for k in range(2):
        md = reference_model(name, k)
        dt = md["dt"]
        n_faces = sum(len(b) for _, b in polys)
        # structure (solverGurobi.cpp:72,:220-230,:241-246,:283-286)
        assert md["offdiag"] == 0 and (md["vtype"][:12 * N] == "C").all()
        assert len(md["vtype"]) == 12 * N + ((N + 1) * P if P else 0) and (md["vtype"][12 * N:] == "B").all()
        assert (md["ind_var"] >= 0).sum() == 4 * N * n_faces
        assert len(md["rhs"]) == 18 * N + 9 + (9 if ff else 6) + 9 * (N - 1) + (N if P else 0) + 4 * N * n_faces
        # the cost: sum over segments and axes of (6 a)^2 (:113-119), nothing on the other coefficients
        q_expect = np.zeros(12 * N)
        q_expect.reshape(N, 12)[:, :3] = 36.0
        assert np.array_equal(md["qdiag"][:12 * N], q_expect)
        sigmas = [rng.integers(0, P, N) for _ in range(3)] if P else [np.zeros(N, int)]
        for sigma in sigmas:
            q, Aeq, beq, Ain, bin_ = sr.model_for_sigma(md if P else dict(md, P=1), sigma)
            Q, Aeq2, beq2, Ain2, bin2 = mf.build(N, pb["x0"], pb["xf"], pb["lim"], dt, polys, sigma, ff)
            assert np.array_equal(np.asarray(Q.todense()).diagonal(), 2.0 * q)
            assert Aeq.shape == Aeq2.shape and np.array_equal(Aeq, Aeq2) and np.array_equal(beq, beq2)
            nb = 18 * N
            assert Ain.shape == Ain2.shape and np.array_equal(Ain[:nb], Ain2[:nb]) and np.array_equal(bin_[:nb], bin2[:nb])
            perm, ofs = [], nb
            for t in range(N):                                   # reference: (face, control point); restatement: (control point, face)
                F = len(polys[int(sigma[t])][1]) if P else 0
                perm += [ofs + cp * F + f for f in range(F) for cp in range(4)]
                ofs += 4 * F
            assert np.array_equal(Ain[nb:], Ain2[perm]) and np.array_equal(bin_[nb:], bin2[perm])


def test_dt_initial_num_samples_and_fill_x_equal_the_reference_code(oracle):
    """fq_dt_initial against the reference's getDTInitial (:659-759: its float temporaries, MinPositiveElement, the max over
    nine times; the polynomial root finder is a stand-in, oracle/stub_eigen), fq_num_samples / fq_fill_x against its resetX /
    fillX (:382-388,:122-168: accumulated sample time, lagging interval index, last sample at rest)."""
    inputs, edge = dt_initial_inputs()
    ref_dt, ref_edge = reference("dt_initial"), reference("dt_initial_edge")
    assert len(ref_dt) == len(inputs) and len(ref_edge) == len(edge)
    n_exact = 0
    for k, (x0, xf, lim, N) in enumerate(inputs):
        a, b = capi.dt_initial(x0, xf, lim, N), ref_dt[k]
        assert a == b or abs(a - b) <= 2e-7 * abs(b), (k, a, b)  # float temporaries: one float ulp at most
        n_exact += a == b
    assert n_exact >= 396
    for (x0, xf, lim, N), b in zip(edge, ref_edge):
        assert capi.dt_initial(x0, xf, lim, N) == b == oracle.dt_initial(x0, xf, lim, N)
    for seed, (N, dt, DC) in enumerate(FILL_X_CASES):
        co = np.random.default_rng(seed).normal(size=(N, 12))
        ref = reference("fill_x.%d" % seed)
        ours = capi.fill_x(N, co, dt, DC)
        assert len(ref) == capi.num_samples(N, dt, DC) == len(ours)
        assert np.abs(ref - ours).max() <= 1e-12 * max(1.0, np.abs(ref).max())
        assert not ref[-1, 3:].any() and not ours[-1, 3:].any()  # :165-167


@pytest.mark.parametrize("N,P,ff", LOOP_CASES)
def test_gen_new_traj_loop_of_the_reference_with_an_independent_solver(oracle, N, P, ff):
    """The reference's genNewTraj (:426-477) compiled from its source, HiGHS + enumeration of the binaries answering optimize():
    the same `solved`, `trials_`, `dt_`, `factor_that_worked_`, coefficients and sampled states as the sweep of the CPU
    restatement (all P^N assignments) and the product's fq_fill_x."""
    n_solved = 0
    for seed in range(3):
        pb, polys = loop_corridor(N, P, ff, seed)
        ref = reference("loop.%d.%d.%d.%d" % (N, P, ff, seed))
        ora = oracle.gen_new_traj(N, pb["x0"], pb["xf"], pb["lim"], polys, 0.01, 1.0, 6.0, 1.0, None, ff)
        assert ref["solved"] == ora["solved"] and ref["trials"] == ora["trials"], (seed, ref["trials"], ora["trials"])
        assert ref["n_optimize"] == ref["trials"]
        assert ref["dt"] == ora["dt"]
        if ref["solved"]:
            n_solved += 1
            assert ref["factor"] == ora["factor"]
            assert np.abs(ref["coeffs"] - ora["coeffs"]).max() <= 1e-6 * max(1.0, np.abs(ora["coeffs"]).max())
            ours = capi.fill_x(N, ora["coeffs"], ora["dt"], 0.01)
            assert ref["n_samples"] == len(ours)                  # the stored states: every 16th and the last
            assert np.abs(ref["samples"] - ours[ref["sample_rows"]]).max() <= 1e-5
    assert n_solved >= 2


def test_reference_loop_refusals(oracle):
    """No factor works: every factor is tried, `solved` is false (:445-472).  StopExecution() before genNewTraj(): no trial at
    all and the flag is reset (:30-39,:445,:474) -- what tests/test_shim_cpu.py asserts of the drop-in class."""
    N, ff = 4, True
    pb, far = refusal_corridor()
    ref = reference("refusal.far")
    ora = oracle.gen_new_traj(N, pb["x0"], far, pb["lim"], pb["polys"], 0.01, 1.0, 3.0, 1.0, None, ff)
    assert not ref["solved"] and not ora["solved"] and ref["trials"] == 3 == ora["trials"] and ref["n_optimize"] == 3
    stopped = reference("refusal.stopped")
    assert not stopped["solved"] and stopped["trials"] == 0 and stopped["n_optimize"] == 0


def test_cpu_restatement_matches_the_committed_reference_sweeps(oracle):
    """tests/golden/reference_sweeps.json holds what THE REFERENCE'S OWN genNewTraj returned (compiled from the original
    project, HiGHS answering optimize(); tools/make_reference_sweep_goldens.py).  The CPU restatement's sweep -- the checker of
    the CUDA path in the GPU tests -- reproduces it: solved, trials_, dt_, factor_that_worked_, coefficients, the sample count and
    the first and last sampled state."""
    import json
    fx = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_sweeps.json")))
    n_solved = n_unsolved = 0
    for c in fx["cases"]:
        polys = [(np.array(p["A"]), np.array(p["b"])) for p in c["polys"]]
        o = oracle.gen_new_traj(c["N"], c["x0"], c["xf"], c["lim"], polys, c["DC"], *c["window"], None, c["force_final"])
        assert o["solved"] == c["solved"] and o["trials"] == c["trials"] and o["dt"] == c["dt"], (c["N"], c["P"], o["trials"], c["trials"])
        if not c["solved"]:
            n_unsolved += 1
            continue
        n_solved += 1
        assert o["factor"] == c["factor"]
        co = np.array(c["coeffs"])
        assert np.abs(o["coeffs"] - co).max() <= 1e-6 * max(1.0, np.abs(co).max())
        X = capi.fill_x(c["N"], o["coeffs"], o["dt"], c["DC"])
        assert len(X) == c["n_samples"]
        assert np.abs(X[0] - np.array(c["first_sample"])).max() <= 1e-5 and np.abs(X[-1] - np.array(c["last_sample"])).max() <= 1e-5
    assert n_solved >= 6 and n_unsolved >= 2
