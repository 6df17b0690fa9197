"""kNN parity: the device map against the reference's own ikd-Tree (its recorded answers, tests/reference_tape.py)."""
import numpy as np
import pytest

from fast_lio_b200 import api, synth
from reference_tape import ReferenceTree

pytestmark = pytest.mark.gpu


def _world_queries(pr):
    """Scan points pushed through the prior pose (float32), as h_share_model does."""
    from oracle.bind import lib
    q = np.zeros((len(pr.scan), 4), dtype=np.float32)
    L = lib()
    tmp = np.zeros(3, dtype=np.float32)
    for i in range(len(pr.scan)):
        L.oracle_transform_point(pr.x_prior, np.ascontiguousarray(pr.scan[i, :3]), tmp)
        q[i, :3] = tmp
    return q


@pytest.mark.parametrize("name", ["tiny", "small", "avia_2k_50k"])
def test_knn_matches_reference_ikdtree(problems, name):
    pr = problems(name)
    q = _world_queries(pr)
    ref = ReferenceTree(f"knn_{name}", pr.map_pts)
    rp, rd, rc = ref.knn(q, 5)
    t = api.KdTree(0, 0.5)
    t.Build(pr.map_pts)
    assert t.validnum() == len(pr.map_pts)
    gp, gd, gc = t.Nearest_Search(q, 5)
    assert np.array_equal(gc, rc)
    # bit-exact squared distances (float32, same operation order as ikd_Tree.cpp:1683-1688)
    assert np.array_equal(gd, rd)
    # identical neighbour coordinates and payload wherever distances are not tied
    tie = np.zeros(len(q), dtype=bool)
    tie[:] = (np.diff(rd, axis=1) == 0).any(axis=1)
    assert np.array_equal(gp[~tie], rp[~tie])


def _brute_d2(q, pts):
    return ((q[0] - pts[:, 0]) ** 2 + (q[1] - pts[:, 1]) ** 2) + (q[2] - pts[:, 2]) ** 2      # float32, the reference's order


def _decided_rows(q, pts, rp, rd):
    """Rows whose point list is determined by the reference's own rules (see test_knn_gridded_map_ties)."""
    decided = np.zeros(len(q), dtype=bool)
    inner_tie = np.zeros(len(q), dtype=bool)
    for i in range(len(q)):
        d = np.sort(_brute_d2(q[i], pts))
        assert np.array_equal(rd[i], d[:5])
        same_d = np.abs(np.diff(rd[i])) < 1e-10
        same_dx = same_d & (np.diff(rp[i][:, 0]) == 0)                 # equal distance AND equal x: the heap's order is unspecified
        decided[i] = d[4] != d[5] and not same_dx.any()
        inner_tie[i] = decided[i] and same_d.any()
    return decided, inner_tie


def test_knn_gridded_map_ties():
    """A lattice map makes squared distances tie exactly.  The distances must still be the reference's bit for bit; the
    POINTS must be the reference's wherever the reference's answer is determined by its own rules: candidates within
    1e-10 of each other are ordered by x (PointType_CMP, ikd_Tree.h:102-108).  Rows in which the k-th and the
    (k+1)-th distance tie are decided by the reference's traversal order (first found stays, ikd_Tree.cpp:1088) -- no
    exact search can reproduce that without being the same tree -- and are excluded from the point comparison."""
    rng = np.random.default_rng(17)
    g = np.arange(-6, 6.01, 0.5, dtype=np.float32)
    X, Y, Z = np.meshgrid(g, g, g[:9], indexing="ij")
    pts = np.stack([X.ravel(), Y.ravel(), Z.ravel(), np.arange(X.size, dtype=np.float32)], axis=1).astype(np.float32)
    pts = pts[rng.permutation(len(pts))]
    q = np.zeros((600, 4), dtype=np.float32)
    q[:, :3] = np.round(rng.uniform(-5, 5, (600, 3)) * 8) / 8          # multiples of 0.125: plenty of equidistant neighbours
    q[:300, 0] += rng.uniform(-0.05, 0.05, 300).astype(np.float32)
    ref = ReferenceTree("knn_gridded_map", pts)
    rp, rd, rc = ref.knn(q, 5)
    t = api.KdTree(0, 0.5); t.Build(pts)
    gp, gd, gc = t.Nearest_Search(q, 5)
    assert np.array_equal(gc, rc) and np.array_equal(gd, rd)
    decided, _ = _decided_rows(q, pts, rp, rd)
    assert decided.sum() >= 50
    assert np.array_equal(gp[decided], rp[decided])


def test_knn_planted_ties_are_ordered_by_x():
    """Every query has two mirrored pairs of neighbours (x - a, x + a: exactly equidistant) and a fifth, distinct one:
    the five neighbours are determined, and the reference returns each pair in ascending x (ikd_Tree.h:102-108)."""
    rng = np.random.default_rng(17)
    qs, ps = [], []
    for i in range(12):
        for j in range(12):
            c = np.array([10.0 * i - 60, 10.0 * j - 60, float(rng.integers(-3, 4))])
            qs.append(c)
            a1, a2 = rng.integers(1, 20, 2) / 64.0
            b = rng.integers(-20, 21, (3, 2)) / 64.0
            ps += [c + [-a1, b[0, 0], b[0, 1]], c + [a1, b[0, 0], b[0, 1]], c + [a2, b[1, 0], b[1, 1] + 0.5],
                   c + [-a2, b[1, 0], b[1, 1] + 0.5], c + [b[2, 0], 0.9, b[2, 1]]]
            for k in range(6):
                ps.append(c + rng.uniform(2.0, 4.5, 3) * rng.choice([-1, 1], 3))
    pts = np.zeros((len(ps), 4), dtype=np.float32); pts[:, :3] = np.array(ps, dtype=np.float32); pts[:, 3] = np.arange(len(ps))
    pts = pts[rng.permutation(len(pts))]
    q = np.zeros((len(qs), 4), dtype=np.float32); q[:, :3] = np.array(qs, dtype=np.float32)
    ref = ReferenceTree("knn_planted_ties", pts)
    rp, rd, rc = ref.knn(q, 5)
    decided, inner_tie = _decided_rows(q, pts, rp, rd)
    assert inner_tie.sum() >= 100                                       # the x rule is exercised
    t = api.KdTree(0, 0.5); t.Build(pts)
    for cell_dir in (True, False):                                      # both search routes obey it
        if not cell_dir:
            t = api.KdTree(0, 0.5, cell_directory=False); t.Build(pts)
        gp, gd, gc = t.Nearest_Search(q, 5)
        assert np.array_equal(gc, rc) and np.array_equal(gd, rd)
        assert np.array_equal(gp[decided], rp[decided])


def test_knn_far_and_crowded_queries_take_the_bvh_route():
    """The cell directory proves most queries exact; queries far from the map and cells holding more points than a
    directory entry lists must come back from the BVH walk with the same exact answer."""
    rng = np.random.default_rng(23)
    dense = rng.uniform(-1, 1, (4000, 4)).astype(np.float32)                     # ~60 points per 1 m cell: crowded
    sparse = rng.uniform(-60, 60, (3000, 4)).astype(np.float32)                  # < 1 point per 100 cells: nothing nearby
    pts = np.concatenate([dense, sparse + np.float32([0, 0, 200, 0])])
    q = np.concatenate([rng.uniform(-2, 2, (200, 4)), rng.uniform(-80, 80, (200, 4)) + [0, 0, 200, 0],
                        rng.uniform(-500, 500, (100, 4))]).astype(np.float32)
    t = api.KdTree(0, 0.5); t.Build(pts)
    gp, gd, gc = t.Nearest_Search(q, 5)
    assert (gc == 5).all()
    for i in range(len(q)):
        assert np.array_equal(gd[i], np.sort(_brute_d2(q[i], pts))[:5])


def test_knn_fewer_than_k_points():
    t = api.KdTree(0, 0.5)
    pts = np.array([[0, 0, 0, 1], [1, 0, 0, 2], [0, 1, 0, 3]], dtype=np.float32)
    t.Build(pts)
    gp, gd, gc = t.Nearest_Search(np.array([[0.1, 0, 0, 0]], dtype=np.float32), 5)
    assert gc[0] == 3
    assert np.allclose(gp[0, 0], [0, 0, 0, 1])
    assert np.isinf(gd[0, 3:]).all()


def test_knn_empty_map():
    t = api.KdTree(0, 0.5)
    gp, gd, gc = t.Nearest_Search(np.zeros((4, 4), dtype=np.float32), 5)
    assert (gc == 0).all()
    t.Build(np.zeros((0, 4), dtype=np.float32))
    gp, gd, gc = t.Nearest_Search(np.zeros((4, 4), dtype=np.float32), 5)
    assert (gc == 0).all() and t.validnum() == 0


def test_knn_brute_force_random():
    rng = np.random.default_rng(5)
    pts = rng.uniform(-20, 20, size=(5000, 4)).astype(np.float32)
    q = rng.uniform(-25, 25, size=(300, 4)).astype(np.float32)
    t = api.KdTree(0, 0.5)
    t.Build(pts)
    gp, gd, gc = t.Nearest_Search(q, 5)
    for i in range(len(q)):
        d = ((q[i, 0] - pts[:, 0]) ** 2 + (q[i, 1] - pts[:, 1]) ** 2) + (q[i, 2] - pts[:, 2]) ** 2   # float32, same order
        order = np.argsort(d, kind="stable")[:5]
        assert np.array_equal(gd[i], d[order])


def test_handles_may_be_destroyed_in_any_order(problems):
    """The C ABI keeps a map alive while a filter or a scan front end created on it exists (Python's cyclic GC may
    finalise the wrappers in any order; a C++ caller's static destructors may too)."""
    import ctypes as C
    pr = problems("tiny")
    L = api.load()
    m, f, s = C.c_void_p(), C.c_void_p(), C.c_void_p()
    assert L.fl_map_create(C.byref(m), 0, 0.5) == 0
    assert L.fl_map_build(m, pr.map_pts, len(pr.map_pts)) == 0
    assert L.fl_filter_create(C.byref(f), m, 1000) == 0
    assert L.fl_scan_create(C.byref(s), m) == 0
    assert L.fl_map_destroy(m) == 0                      # the caller lets go first
    x = pr.x_prior.copy(); P = pr.P_prior.copy()
    assert L.fl_filter_update(f, pr.scan, len(pr.scan), x, P, pr.R, None) == 0      # the filter still has its map
    assert L.fl_filter_destroy(f) == 0
    assert L.fl_scan_destroy(s) == 0
    t = api.KdTree(0, 0.5); t.Build(pr.map_pts)           # and nothing is left pending in the CUDA error state
    assert t.validnum() == len(pr.map_pts)
