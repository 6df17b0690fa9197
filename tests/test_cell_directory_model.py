"""CPU: the cell-directory model returns the exact k-NN (same distances as a brute-force float32 search and as the
reference's ikd-Tree) and settles within the 27-cell neighbourhood for almost every query of the benchmark scene."""
import os

import numpy as np
import pytest

from fast_lio_b200 import synth
from cell_directory_model import CellDirectoryModel
from test_oracle_golden import GOLD, world_queries


def brute(pts, q, k=5):
    d = q[None, :3].astype(np.float32) - pts[:, :3]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).astype(np.float32) + d[:, 2] * d[:, 2]
    order = np.argsort(d2, kind="stable")[:k]
    return order, d2[order].astype(np.float32)


@pytest.mark.parametrize("cell", [0.5, 1.0, 2.0])
def test_rings_give_the_exact_knn(problems, cell):
    pr = problems("small")
    m = CellDirectoryModel(pr.map_pts, cell)
    q = world_queries(pr)[::25]
    rings = []
    for qq in q:
        idx, d2, r, _ = m.knn(qq)
        bi, bd = brute(pr.map_pts, qq)
        assert np.array_equal(d2, bd)
        assert set(idx.tolist()) == set(bi.tolist())
        rings.append(r)
    if cell >= 1.0:
        assert np.mean(np.array(rings) <= 1) > 0.95      # the 27-cell neighbourhood settles almost every query


def test_model_matches_reference_ikdtree(problems):
    pr = problems("tiny")
    m = CellDirectoryModel(pr.map_pts, 1.0)
    g = np.load(os.path.join(GOLD, "tiny.npz"))                 # the reference's kNN of these queries (tests/golden/make_golden.py)
    q = world_queries(pr)[:200]
    d_ref, cnt = g["knn_d2"][:200], g["knn_cnt"][:200]
    for i, qq in enumerate(q):
        _, d2, _, _ = m.knn(qq)
        assert cnt[i] == 5 and np.array_equal(d2, d_ref[i])


def test_sparse_and_degenerate_maps():
    pts = np.array([[0, 0, 0, 1], [10, 0, 0, 2], [0, 10, 0, 3]], np.float32)     # fewer than k points: rings stop at the map's extent
    m = CellDirectoryModel(pts, 1.0)
    idx, d2, r, _ = m.knn(np.array([1.0, 1.0, 0.0], np.float32))
    assert len(idx) == 3 and np.array_equal(d2, np.array([2.0, 82.0, 82.0], np.float32))
    far = CellDirectoryModel(np.array([[20.5, 0.2, 0.1, 1]] * 5, np.float32) + np.arange(5, dtype=np.float32)[:, None] * 0.01, 1.0)
    idx, d2, r, _ = far.knn(np.zeros(3, np.float32))
    assert len(idx) == 5 and r >= 19                    # a far query walks rings until it reaches the points
    empty = CellDirectoryModel(np.zeros((0, 4), np.float32), 1.0)
    assert len(empty.knn(np.zeros(3, np.float32))[0]) == 0


@pytest.mark.parametrize("cell", [0.3, 0.7, 1.0])
def test_halo_rule_never_claims_a_wrong_answer(cell):
    """The product's proof rule (map.cuh cell_knn) with its float32 cell arithmetic: whatever it declares exact IS the brute-force
    answer, also for points and queries sitting within rounding of the cell faces and far from the origin, where fl(x * fl(1/cell))
    can file a point one cell off."""
    from cell_directory_model import HaloRuleModel
    rng = np.random.default_rng(7)
    f = np.float32
    origin = np.array([350, -200, 40], np.int64)                                          # cells; far from the origin: coarse ulps
    n = 300                                                                               # sparse enough that the fifth distance is near the proven radius (a rule 0.3 cell too generous fails here)
    cellidx = origin[None, :] + rng.integers(0, 5, size=(n, 3))
    pts3 = ((cellidx + rng.uniform(0, 1, size=(n, 3))) * float(cell)).astype(np.float32)     # uniform in a 5x5x5 block of cells ...
    axis = rng.integers(0, 3, size=n)
    onface = (cellidx[np.arange(n), axis] * f(cell)).astype(np.float32)
    ulp = np.spacing(np.abs(onface)).astype(np.float32)
    sel = rng.uniform(size=n) < 0.5
    pts3[np.arange(n)[sel], axis[sel]] = (onface + ulp * rng.integers(-3, 4, size=n).astype(np.float32))[sel]   # ... half of them within 3 ulps of a face
    pts = np.concatenate([pts3, np.zeros((n, 1), np.float32)], axis=1).astype(np.float32)
    near = pts3[sel]
    m = HaloRuleModel(pts, cell)
    # queries: on / next to faces that have points around them, and at random offsets inside those cells
    base = near[rng.integers(0, len(near), size=400)]
    q = np.concatenate([base, base + np.spacing(np.abs(base)).astype(np.float32),
                        base + rng.uniform(-0.5, 0.5, size=base.shape).astype(np.float32) * f(cell)], axis=0).astype(np.float32)
    proven = 0
    for qq in q:
        idx, d2, ok = m.knn(qq)
        if not ok:
            continue
        proven += 1
        bi, bd = brute(pts, qq)
        assert np.array_equal(d2, bd), (qq, d2, bd)
    assert proven > 50          # the rule must be exercised, not vacuous


def test_halo_rule_on_the_benchmark_scene(problems):
    from cell_directory_model import HaloRuleModel
    pr = problems("small")
    m = HaloRuleModel(pr.map_pts, 1.0)
    q = world_queries(pr)[::10]
    ok_n = 0
    for qq in q:
        idx, d2, ok = m.knn(qq)
        if ok:
            ok_n += 1
            bi, bd = brute(pr.map_pts, qq)
            assert np.array_equal(d2, bd)
    assert ok_n > 0.9 * len(q)       # almost every query of the scene is settled by its cell's halo list alone


def misfiled_points(cell):
    """x just below a cell face k*cell that the float32 filing floor(fl(x * fl(1/cell))) nevertheless puts into cell k"""
    f = np.float32
    c = f(cell)
    inv = f(1) / c
    out = []
    for k in range(-400, 400):
        x = np.nextafter(f(k) * c, f(-np.inf), dtype=np.float32)
        if np.floor(f(x * inv)) >= k and float(x) < k * float(c):
            out.append((k, x))
    return out


@pytest.mark.parametrize("cell", [0.3, 0.7])
def test_margin_covers_points_filed_one_cell_off(cell):
    """A point P geometrically inside the 3x3x3 block but FILED in the next cell (float32 rounding of x/cell) is missing from
    the halo list.  With a fifth candidate a hair farther than P, the naive rule (no margin) declares the wrong five exact;
    the product's margin withholds the proof, and the query goes to the BVH walk."""
    from cell_directory_model import HaloRuleModel
    f = np.float32
    c = f(cell)
    cases = misfiled_points(cell)
    assert cases, "float32 filing has no rounding cases for this cell size?"
    naive_wrong = 0
    for k, xp in cases:
        j = k - 2                                              # the query's cell: its block ends at the face k*cell
        qx = f((j + 0.55) * float(c))
        qy = qz = f(0.5) * c
        P = np.array([xp, qy, qz], np.float32)
        dP = f(xp - qx)
        g_naive = f(f(f(j + 1) * c - qx) + c)
        if not dP < g_naive:
            continue
        d5 = f((float(dP) + float(g_naive)) / 2)
        close = [[qx + f(0.01) * c * f(i + 1), qy, qz] for i in range(4)]
        pts3 = np.array(close + [[qx, qy + d5, qz], list(P)], np.float32)
        pts = np.concatenate([pts3, np.zeros((len(pts3), 1), np.float32)], axis=1)
        q = np.array([qx, qy, qz], np.float32)
        _, bd = brute(pts, q)
        idx, d2, ok = HaloRuleModel(pts, cell).knn(q)
        assert (not ok) or np.array_equal(d2, bd)                  # the product rule: never a wrong claim
        idx, d2, ok = HaloRuleModel(pts, cell, marg_scale=0.0).knn(q)
        naive_wrong += bool(ok and not np.array_equal(d2, bd))
    assert naive_wrong > 0           # the margin is load-bearing: without it these constructions are answered wrongly
