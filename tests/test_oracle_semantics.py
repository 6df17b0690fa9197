"""CPU: pin the oracle pieces against each other and against the reference's own ikd-Tree (its recorded answers)."""
import numpy as np
import pytest

from fast_lio_b200 import synth
from oracle import bind
from reference_tape import ReferenceTree
from semantics import VoxelMapModel, sort_rows


def test_port_knn_equals_reference_ikdtree(problems):
    pr = problems("small")
    q = pr.map_pts[::7].copy()
    q[:, :3] += 0.21
    a = ReferenceTree("port_knn_small", pr.map_pts)
    b = bind.KdTree(pr.map_pts, "port")
    pa, da, ca = a.knn(q)
    pb, db, cb = b.knn(q)
    assert np.array_equal(ca, cb) and np.array_equal(da, db) and np.array_equal(pa, pb)


def test_knn_port_brute_force():
    rng = np.random.default_rng(0)
    pts = rng.uniform(-10, 10, (3000, 4)).astype(np.float32)
    q = rng.uniform(-12, 12, (200, 4)).astype(np.float32)
    t = bind.KdTree(pts, "port")
    p, d, c = t.knn(q)
    for i in range(len(q)):
        dd = ((q[i, 0] - pts[:, 0]) ** 2 + (q[i, 1] - pts[:, 1]) ** 2) + (q[i, 2] - pts[:, 2]) ** 2
        assert np.array_equal(d[i], np.sort(dd)[:5])


def test_mutation_model_equals_reference_ikdtree():
    rng = np.random.default_rng(4)
    pts = rng.uniform(-4, 4, (2500, 4)).astype(np.float32)
    r = ReferenceTree("mutation_model", pts, downsample=0.5)
    m = VoxelMapModel(pts, 0.5)
    for rep in range(3):
        batch = rng.uniform(-5, 5, (700, 4)).astype(np.float32)
        assert r.add(batch, True) == m.add_points(batch, True)
        assert np.array_equal(sort_rows(r.flatten()), sort_rows(m.flatten()))
        box = np.array([[-1.0 + rep, -2, -2, 0.5 + rep, 2, 2]], dtype=np.float32)
        assert r.delete_boxes(box) == m.delete_boxes(box)
        assert np.array_equal(sort_rows(r.flatten()), sort_rows(m.flatten()))
        extra = rng.uniform(-5, 5, (100, 4)).astype(np.float32)
        assert r.add(extra, False) == m.add_points(extra, False) == 0
    assert r.validnum() == len(m.flatten())
