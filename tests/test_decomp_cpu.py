"""Host-side convex decomposition (fq_ellipsoid_decomp, faster_b200/csrc/fq_decomp.cpp) against
  * the REFERENCE'S OWN CODE: DecompUtil's EllipsoidDecomp3D compiled unmodified from the original project (oracle/Makefile ->
    oracle/_ref/libdecomp_ref.so; oracle/stub_eigen supplies the small-matrix arithmetic Eigen would), driven like
    JPS_Manager::cvxEllipsoidDecomp (oracle/decomp_ref_wrap.cpp) -- the pinned oracle of this path.  What it returned on the
    inputs below is stored in tests/golden/reference_decomp.npz (tools/make_reference_goldens.py);
  * the numpy restatement of the same (oracle/decomp_oracle.py), itself checked against the compiled reference here, in the
    reference's row order."""
import functools
import os

import numpy as np
import pytest

from faster_b200 import capi, corridor as cr
from oracle import decomp_oracle as do

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_decomp.npz")
DEMO_PATH = np.array([[5, 11.5, 0.5], [13, 11.5, 3.0], [14, 10.5, 1.5], [14, 5, 2.5]], float)        # path3d.txt
EDGE_CASES = [
    (np.array([[0.0, 0.0, 1.0], [1.2, 0.3, 1.1]]), np.zeros((0, 3)), 0.42),
    (np.array([[0.0, 0.0, 0.5], [0.0, 0.0, 1.6]]), np.array([[1.0, 0.2, 1.0], [-0.8, -0.9, 0.7], [2.0, 0.0, 1.0], [0.3, 1.1, 1.4], [5.0, 5.0, 5.0]]), 0.2),
    (np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 1.0]]), np.array([[2.5, 0.0, 1.0], [-1.5, 0.0, 1.0], [0.5, 2.0, 1.0], [0.5, -2.0, 1.0], [0.5, 0.0, 2.0]]), 0.0),
    (np.array([[0.0, 0.0, 1.0], [1.0, 1.0, 1.2]]), np.array([[0.4, 1.3, 1.0]] * 3 + [[1.2, -0.4, 1.1]] * 2), 0.1),
]


@functools.lru_cache(maxsize=None)
def reference(key):
    """The reference's polytopes stored under `key`, one list of (A, b) per call, in call order."""
    with np.load(GOLDEN) as z:
        Ab, rows, polys = z[key + ".Ab"], z[key + ".rows"], z[key + ".polys"]
    ends = np.cumsum(rows)
    flat = [(Ab[e - n:e, :3], Ab[e - n:e, 3]) for n, e in zip(rows, ends)]
    cuts = np.concatenate([[0], np.cumsum(polys)])
    return [flat[a:b] for a, b in zip(cuts[:-1], cuts[1:])]


def _same(polys_a, polys_b, tol=1e-9):
    """Same faces.  The order of the obstacle-derived faces may differ where two obstacle points are equidistant from
    the ellipsoid to the last bit (regularly sampled cylinders produce such ties; the product evaluates C^-1 in closed
    form, the oracle inverts C numerically), so rows are compared as sorted sets; the six bounding-box faces and the
    ground face must sit at the end in the reference's order."""
    assert len(polys_a) == len(polys_b)
    for (A1, b1), (A2, b2) in zip(polys_a, polys_b):
        assert A1.shape == A2.shape, "face counts differ"
        assert np.abs(A1[-7:] - A2[-7:]).max() <= tol and np.abs(b1[-7:] - b2[-7:]).max() <= tol
        r1 = np.hstack([A1, b1[:, None]])
        r2 = np.hstack([A2, b2[:, None]])
        r1 = r1[np.lexsort(np.round(r1, 7).T[::-1])]
        r2 = r2[np.lexsort(np.round(r2, 7).T[::-1])]
        assert np.abs(r1 - r2).max() <= tol


@pytest.mark.parametrize("seed", range(6))
def test_forest_decomposition_matches_oracle(built_lib, seed):
    obs, centres, radii = cr.make_forest(40 + seed)
    path = cr.forest_path(140 + seed, centres, radii, 4, clearance=0.42 * 1.45 + 0.05)
    a = capi.ellipsoid_decomp(path, obs, (2.0, 2.0, 1.0), 0.42, 0.0)
    b = do.cvx_ellipsoid_decomp(path, obs, (2.0, 2.0, 1.0), 0.42, 0.0)
    _same(a, b)
    for k, (A, bb) in enumerate(a):
        # conventions the solver relies on (SURVEY Appendix B): unit normals, segment inside, bbox + ground faces last
        assert np.allclose(np.linalg.norm(A, axis=1), 1.0, atol=1e-12)
        for p in (path[k], path[k + 1], 0.5 * (path[k] + path[k + 1])):
            assert (A @ p - bb).max() <= 1e-9
        assert np.array_equal(A[-1], [0.0, 0.0, -1.0]) and bb[-1] == 0.0
        assert len(bb) >= 7
        # no (inflated) obstacle point is strictly inside the polytope: every kept point is cut by some face
        inside = np.all(obs @ A.T - bb < -0.42 * 1.8, axis=1)
        assert not inside.any()


def test_edge_inputs(built_lib):
    path = np.array([[0.0, 0.0, 1.0], [1.2, 0.3, 1.1]])
    # no obstacles at all: only the six bbox faces and the ground face
    a = capi.ellipsoid_decomp(path, np.zeros((0, 3)))
    b = do.cvx_ellipsoid_decomp(path, np.zeros((0, 3)))
    _same(a, b)
    assert len(a[0][1]) == 7
    # a vertical segment (dir_h degenerates, line_segment.h:64-70) and obstacles exactly on a bbox face
    path = np.array([[0.0, 0.0, 0.5], [0.0, 0.0, 1.6]])
    obs = np.array([[1.0, 0.2, 1.0], [-0.8, -0.9, 0.7], [2.0, 0.0, 1.0], [0.3, 1.1, 1.4], [5.0, 5.0, 5.0]])
    _same(capi.ellipsoid_decomp(path, obs, inflate=0.2), do.cvx_ellipsoid_decomp(path, obs, inflate=0.2))
    # capacity too small -> error code, not a crash
    with pytest.raises(capi.FqError):
        capi.ellipsoid_decomp(np.array([[0.0, 0, 1], [1, 0, 1]]), np.zeros((0, 3)), cap_rows=3)


def test_random_clouds(built_lib):
    rng = np.random.default_rng(9)
    for k in range(25):
        p1 = rng.uniform(-2, 2, 3)
        p2 = p1 + rng.uniform(-1.5, 1.5, 3)
        if np.linalg.norm(p2 - p1) < 0.3:
            continue
        mid = 0.5 * (p1 + p2)
        obs = mid + rng.normal(size=(int(rng.integers(1, 200)), 3)) * rng.uniform(0.5, 2.5)
        d = np.linalg.norm(np.cross(obs - p1, obs - p2), axis=1) / np.linalg.norm(p2 - p1)
        obs = obs[d > 0.6]                       # keep the segment itself obstacle-free
        _same(capi.ellipsoid_decomp(np.array([p1, p2]), obs, inflate=0.2), do.cvx_ellipsoid_decomp(np.array([p1, p2]), obs, inflate=0.2))


def test_bbox_faces_reproduce_the_reference_demo_polytopes(built_lib, demo_corridor):
    """Reference-held OUTPUTS of the decomposition: the three polytopes hard-coded in faster/other/gurobi_continuous.cpp
    (:318-401; extracted to tests/golden/corridor_continuous.json) are what DecompUtil's EllipsoidDecomp3D produced for
    thirdparty/DecompROS/decomp_test_node/data/path3d.txt with the demo's local bounding box (1, 2, 1)
    (decomp_test_node/src/test_path_decomp_3d.cpp:43).  Their last six rows are the local-bbox faces (line_segment.h:57-98),
    which depend on the path alone -- the product's fq_ellipsoid_decomp must reproduce them, in the reference's order and
    with its signs, to the six digits the demo prints.  Their first rows come from the demo's obstacle cloud (a ROS bag,
    not reproducible here); for those, the convention the solver relies on is checked: A x <= b holds along the segment."""
    path = np.array([[5, 11.5, 0.5], [13, 11.5, 3.0], [14, 10.5, 1.5], [14, 5, 2.5]], float)      # path3d.txt
    ours = capi.ellipsoid_decomp(path, np.zeros((0, 3)), (1.0, 2.0, 1.0), 0.0, -100.0)
    for k, (A, b) in enumerate(demo_corridor["polys"]):
        Ao, bo = ours[k]
        assert Ao.shape[0] == 7                                   # six bbox faces + the ground face (jps_manager.cpp:118-122)
        assert np.abs(A[-6:] - Ao[:6]).max() < 5e-5 and np.abs(b[-6:] - bo[:6]).max() < 5e-5
        assert np.allclose(np.linalg.norm(A, axis=1), 1.0, atol=2e-5)          # unit normals (ellipsoid.h:65-73)
        for s in np.linspace(0.0, 1.0, 11):
            p = path[k] + s * (path[k + 1] - path[k])
            assert (A @ p - b).max() < 0.0                        # the segment is strictly inside the reference's polytope
        # obstacle-derived faces keep the segment at least an obstacle-inflation away... they are cut planes, not bbox:
        assert (A[:-6] @ (0.5 * (path[k] + path[k + 1])) - b[:-6]).max() < -0.1


def test_decomposition_properties_independent_of_both_implementations(built_lib):
    """What must hold for ANY correct decomposition (decomp_base.h:83-115, line_segment.h:156-252), checked on the product's
    output without reference to the oracle: the segment is inside its polytope; every obstacle point inside the local
    bounding box is outside or on at least one face once the face is pushed out by the inflation radius; faces are unit
    normals; the bbox and ground faces close the polytope."""
    r = 0.42
    for seed in range(8):
        obs, centres, radii = cr.make_forest(300 + seed)
        path = cr.forest_path(400 + seed, centres, radii, 3, clearance=r * 1.45 + 0.05)
        polys = capi.ellipsoid_decomp(path, obs, (2.0, 2.0, 1.0), r, 0.0)
        for k, (A, b) in enumerate(polys):
            assert np.allclose(np.linalg.norm(A, axis=1), 1.0, atol=1e-12)
            for s in np.linspace(0, 1, 9):
                assert (A @ (path[k] + s * (path[k + 1] - path[k])) - b).max() <= 1e-9
            # obstacle points well inside the six bbox faces and above the ground:
            box_in = np.all(obs @ A[-7:].T - b[-7:] < -1e-9, axis=1)
            pts = obs[box_in]
            if len(pts):
                # each of them is excluded by an obstacle face, up to the inflation radius
                excl = (pts @ A[:-7].T - b[:-7]).max(axis=1) if A.shape[0] > 7 else np.full(len(pts), -np.inf)
                assert (excl >= -r - 1e-9).all(), (seed, k, excl.min())


def _clouds(seed, n):
    """Random paths of 1-3 segments inside random clouds, and forest corridors (the config-4 generator)."""
    rng = np.random.default_rng(seed)
    for k in range(n):
        if k % 3 == 2:
            obs, centres, radii = cr.make_forest(700 + seed * 50 + k)
            yield cr.forest_path(800 + seed * 50 + k, centres, radii, 3, clearance=0.42 * 1.45 + 0.05), obs, 0.42
        else:
            npts = int(rng.integers(2, 5))
            path = np.cumsum(rng.uniform(-1.5, 1.5, (npts, 3)) * [1, 1, 0.3], axis=0) + [0, 0, 1.0]
            if min(np.linalg.norm(np.diff(path, axis=0), axis=1)) < 0.2:
                continue
            obs = rng.uniform(-4, 4, (int(rng.integers(0, 500)), 3)) * [1, 1, 0.5] + [0, 0, 1.0]
            yield path, obs, float(rng.choice([0.0, 0.2, 0.42]))


def test_product_matches_the_reference_code(built_lib):
    """fq_ellipsoid_decomp against DecompUtil itself (compiled from the reference tree): the same faces to 1e-9, the six
    bounding-box faces and the ground face last and in the reference's order.  The two obstacle points the final ellipsoid
    touches are at distance 1 from it up to rounding, so the reference's first two faces may come out in either order
    (it inverts C numerically, the product keeps C^-1 in closed form): obstacle faces are compared as sets."""
    n_poly = n_rows = in_order = 0
    clouds = list(_clouds(1, 45))
    assert len(clouds) == len(reference("product"))
    for (path, obs, r), ref in zip(clouds, reference("product")):
        ours = capi.ellipsoid_decomp(path, obs, (2.0, 2.0, 1.0), r, 0.0)
        _same(ours, ref)
        for (A1, b1), (A2, b2) in zip(ours, ref):
            n_poly += 1
            n_rows += len(b1)
            in_order += int(np.abs(A1 - A2).max() <= 1e-9 and np.abs(b1 - b2).max() <= 1e-9)
    assert n_poly >= 60 and n_rows >= 700
    assert in_order >= 0.7 * n_poly                     # and most polytopes agree row by row as well


def test_numpy_restatement_matches_the_reference_code():
    """oracle/decomp_oracle.py (the checker the other tests of this file use on inputs without stored reference outputs)
    against the compiled reference: the same faces; and row by row in most polytopes (it inverts C numerically like the
    reference; regularly sampled cylinders still produce exact distance ties)."""
    n_poly = in_order = 0
    clouds = list(_clouds(2, 30))
    assert len(clouds) == len(reference("restatement"))
    for (path, obs, r), ref in zip(clouds, reference("restatement")):
        mine = do.cvx_ellipsoid_decomp(path, obs, (2.0, 2.0, 1.0), r, 0.0)
        _same(mine, ref)
        for (A1, b1), (A2, b2) in zip(mine, ref):
            n_poly += 1
            in_order += int(np.abs(A1 - A2).max() <= 1e-9 and np.abs(b1 - b2).max() <= 1e-9)
    assert n_poly >= 40 and in_order >= 0.8 * n_poly, (n_poly, in_order)


def test_reference_code_reproduces_the_demo_polytopes_bbox_rows(demo_corridor):
    """The compiled reference on the demo's own path (decomp_test_node/data/path3d.txt, local bbox (1, 2, 1)) reproduces the
    six bounding-box rows of the polytopes printed in faster/other/gurobi_continuous.cpp:318-401 -- the wrapper and the Eigen
    stand-in drive the reference's code the way the reference's demo did."""
    ref = reference("demo")[0]
    for k, (A, b) in enumerate(demo_corridor["polys"]):
        Ar, br = ref[k]
        assert Ar.shape[0] == 7
        assert np.abs(A[-6:] - Ar[:6]).max() < 5e-5 and np.abs(b[-6:] - br[:6]).max() < 5e-5


def test_reference_edge_cases_agree(built_lib):
    """No obstacles; a vertical segment (dir_h degenerates, line_segment.h:64-70); points exactly on a bounding-box face;
    a point on the segment's axis beyond its ends; duplicate points."""
    assert len(reference("edge")) == len(EDGE_CASES)
    for (path, obs, r), ref in zip(EDGE_CASES, reference("edge")):
        _same(capi.ellipsoid_decomp(path, obs, inflate=r), ref)
