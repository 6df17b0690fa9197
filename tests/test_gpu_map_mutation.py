"""Add_Points / Delete_Point_Boxes parity of the device map against the reference's ikd-Tree."""
import numpy as np
import pytest

from fast_lio_b200 import api, synth
from reference_tape import ReferenceTree
from semantics import VoxelMapModel, sort_rows

pytestmark = pytest.mark.gpu


def make_batch(rng, base_pts, n, spread=0.3, far_frac=0.2):
    """New points: most near existing map points (compete in their voxel), some in fresh space."""
    idx = rng.integers(0, len(base_pts), n)
    b = base_pts[idx].copy()
    b[:, :3] += rng.normal(0, spread, (n, 3)).astype(np.float32)
    far = rng.random(n) < far_frac
    b[far, :3] += rng.uniform(5, 30, (int(far.sum()), 3)).astype(np.float32)
    b[:, 3] = rng.uniform(100, 200, n).astype(np.float32)
    return np.ascontiguousarray(b.astype(np.float32))


def check_same_map(g: api.KdTree, r, queries):
    gf, rf = sort_rows(g.flatten()), sort_rows(r.flatten())
    assert g.validnum() == r.validnum() == len(rf)
    assert np.array_equal(gf, rf)
    gp, gd, gc = g.Nearest_Search(queries, 5)
    rp, rd, rc = r.knn(queries, 5)
    assert np.array_equal(gc, rc)
    assert np.array_equal(gd, rd)


@pytest.mark.parametrize("name", ["tiny", "small"])
def test_delete_boxes(problems, name):
    pr = problems(name)
    rng = np.random.default_rng(11)
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    r = ReferenceTree(f"delete_boxes_{name}", pr.map_pts)
    q = make_batch(rng, pr.map_pts, 256)
    lo = pr.map_pts[:, :3].min(0); hi = pr.map_pts[:, :3].max(0)
    for rep in range(3):
        c = rng.uniform(lo, hi)
        half = rng.uniform(1.0, 8.0, 3)
        boxes = np.array([[*(c - half), *(c + half)], [*(c + 3), *(c + 3 + half)]], dtype=np.float32)
        assert g.Delete_Point_Boxes(boxes) == r.delete_boxes(boxes)
        check_same_map(g, r, q)
    # deleting the same boxes again removes nothing
    assert g.Delete_Point_Boxes(boxes) == 0


def test_delete_half_open_boundaries():
    pts = np.array([[0, 0, 0, 1], [1, 0, 0, 2], [0.5, 0.5, 0.5, 3], [1, 1, 1, 4]], dtype=np.float32)
    g = api.KdTree(0, 0.5); g.Build(pts)
    # [0,1) x [0,1) x [0,1): contains (0,0,0) and (.5,.5,.5); excludes x == 1
    assert g.Delete_Point_Boxes(np.array([[0, 0, 0, 1, 1, 1]], dtype=np.float32)) == 2
    left = sort_rows(g.flatten())
    assert np.array_equal(left[:, 3], [2, 4])


@pytest.mark.parametrize("name", ["tiny", "small"])
def test_add_points_downsample(problems, name):
    pr = problems(name)
    rng = np.random.default_rng(7)
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    r = ReferenceTree(f"add_points_downsample_{name}", pr.map_pts)
    q = make_batch(rng, pr.map_pts, 256)
    for rep in range(4):
        batch = make_batch(rng, pr.map_pts, 1500)
        assert g.Add_Points(batch, True) == r.add(batch, True)
        check_same_map(g, r, q)


def test_add_points_no_downsample(problems):
    pr = problems("tiny")
    rng = np.random.default_rng(9)
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    r = ReferenceTree("add_points_no_downsample", pr.map_pts)
    q = make_batch(rng, pr.map_pts, 128)
    batch = make_batch(rng, pr.map_pts, 2000)
    assert g.Add_Points(batch, False) == r.add(batch, False) == 0
    check_same_map(g, r, q)


def test_add_into_non_downsampled_map_and_model():
    """Build() does not downsample: voxels may hold many points; the first touch collapses them."""
    rng = np.random.default_rng(3)
    pts = rng.uniform(-3, 3, (3000, 4)).astype(np.float32)       # ~14 points per 0.5 m voxel
    batch = rng.uniform(-3.5, 3.5, (800, 4)).astype(np.float32)
    g = api.KdTree(0, 0.5); g.Build(pts)
    m = VoxelMapModel(pts, 0.5)
    assert g.Add_Points(batch, True) == m.add_points(batch, True)
    assert np.array_equal(sort_rows(g.flatten()), sort_rows(m.flatten()))
    r = ReferenceTree("add_into_non_downsampled_map", pts)
    r.add(batch, True)
    assert np.array_equal(sort_rows(g.flatten()), sort_rows(r.flatten()))


def test_overflow_chain_and_rebuild():
    """Many inserts into one region exhaust leaf slack, chain overflow leaves, then trigger a re-pack;
    the search stays exact throughout."""
    rng = np.random.default_rng(21)
    pts = rng.uniform(-50, 50, (20000, 4)).astype(np.float32)
    g = api.KdTree(0, 0.5); g.Build(pts)
    allpts = [pts]
    for rep in range(6):
        extra = rng.normal(0, 1.0, (4000, 4)).astype(np.float32) + np.float32(10 * rep)
        assert g.Add_Points(extra, False) == 0
        allpts.append(extra)
        cur = np.concatenate(allpts)
        q = cur[rng.integers(0, len(cur), 200)] + rng.normal(0, 0.05, (200, 4)).astype(np.float32)
        gp, gd, gc = g.Nearest_Search(q, 5)
        for i in range(len(q)):
            d = ((q[i, 0] - cur[:, 0]) ** 2 + (q[i, 1] - cur[:, 1]) ** 2) + (q[i, 2] - cur[:, 2]) ** 2
            assert np.array_equal(gd[i], np.sort(d)[:5])
    st = g.stats()
    assert g.validnum() == len(np.concatenate(allpts))
    assert st["rebuilds"] >= 1 or st["overflow_leaves"] > 0


def test_stream_of_scans_matches_reference(problems):
    """Config-4 style loop on a small map: delete boxes, add with and without downsampling, search."""
    pr = problems("small")
    rng = np.random.default_rng(33)
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    r = ReferenceTree("stream_of_scans_map", pr.map_pts)
    for step in range(5):
        batch = make_batch(rng, pr.map_pts, 800)
        assert g.Add_Points(batch[:600], True) == r.add(batch[:600], True)
        assert g.Add_Points(batch[600:], False) == r.add(batch[600:], False)
        c = np.array([-40.0 + 10 * step, 0, 0])
        box = np.array([[c[0], -100, -10, c[0] + 6, 100, 30]], dtype=np.float32)
        assert g.Delete_Point_Boxes(box) == r.delete_boxes(box)
        check_same_map(g, r, make_batch(rng, pr.map_pts, 200))


def test_acquire_removed_points_and_add_point_boxes(problems):
    """a14 leftovers: acquire_removed_points (ikd_Tree.cpp:661-676) returns what Delete_Point_Boxes removed since the last call;
    Add_Point_Boxes (ikd_Tree.cpp:576-603) brings box-deleted points back -- but not points removed by down-sampling."""
    pr = problems("small")
    rng = np.random.default_rng(41)
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    assert len(g.acquire_removed_points()) == 0                 # starts the record (laserMapping.cpp:273 asks before every delete)
    before = sort_rows(g.flatten())
    c = pr.map_pts[:, :3].mean(0)
    boxes = np.array([[*(c - 6), *(c + 6)], [*(c + 8), *(c + 15)]], dtype=np.float32)
    n_del = g.Delete_Point_Boxes(boxes)
    assert n_del > 0
    after = sort_rows(g.flatten())
    removed = sort_rows(g.acquire_removed_points())
    assert len(removed) == n_del and len(after) == len(before) - n_del
    assert np.array_equal(sort_rows(np.concatenate([after, removed])), before)
    assert len(g.acquire_removed_points()) == 0                 # handed over once
    # down-sampling removes points too: those do not come back
    batch = make_batch(rng, pr.map_pts, 1200, far_frac=0.0)
    g.Add_Points(batch, True)
    mid = sort_rows(g.flatten())
    n_back = g.Add_Point_Boxes(boxes)
    assert 0 < n_back <= n_del
    now = sort_rows(g.flatten())
    assert g.validnum() == len(now) == len(mid) + n_back
    # every revived point is one of the removed ones, and the search sees them again
    keyset = {tuple(r) for r in removed}
    added_back = [r for r in now if tuple(r) in keyset]
    assert len(added_back) == n_back
    q = np.ascontiguousarray(np.array(added_back[:50], dtype=np.float32))
    gp, gd, gc = g.Nearest_Search(q, 1)
    assert (gd[:, 0] == 0).all()
    # without intervening inserts the reference restores the map exactly
    g2 = api.KdTree(0, 0.5); g2.Build(pr.map_pts)
    g2.Delete_Point_Boxes(boxes)
    assert g2.Add_Point_Boxes(boxes) == n_del
    assert np.array_equal(sort_rows(g2.flatten()), before)
    qq = make_batch(rng, pr.map_pts, 200)
    r = ReferenceTree("add_point_boxes", pr.map_pts)
    assert np.array_equal(g2.Nearest_Search(qq, 5)[1], r.knn(qq, 5)[1])


def test_directory_lists_grow_and_slots_are_reused():
    """Inserts fill the halo lists of the cells they touch; a list that runs out of room is made anew from the map (k_halo_fix);
    deleted points' slots are re-used by later inserts (their old listings stay behind).  The search must stay exact throughout."""
    rng = np.random.default_rng(77)

    def voxel_points(n, lo, hi):            # at most one point per 0.5 m voxel, like a down-sampled LiDAR map
        c = np.unique(rng.integers(int(lo / 0.5), int(hi / 0.5), (n, 3)), axis=0)
        p = np.zeros((len(c), 4), dtype=np.float32)
        p[:, :3] = (c + rng.uniform(0.05, 0.45, c.shape)).astype(np.float32) * np.float32(0.5)
        p[:, 3] = rng.uniform(1, 100, len(c)).astype(np.float32)
        return p

    base = voxel_points(3000, -20, 20)
    g = api.KdTree(0, 0.5); g.Build(base)
    cur = {tuple(r) for r in base}
    for rep in range(12):
        batch = voxel_points(2500, -12, 12)                                   # keeps hitting the same cells: their lists fill up
        g.Add_Points(batch, False)
        cur |= {tuple(r) for r in batch}
        if rep % 3 == 2:                                                      # delete a slab, then refill it: slots get re-used
            box = np.array([[-6.0, -30, -30, 0.0, 30, 30]], dtype=np.float32)
            g.Delete_Point_Boxes(box)
            cur = {r for r in cur if not (-6.0 <= r[0] < 0.0)}
        pts = np.array(sorted(cur), dtype=np.float32)
        assert g.validnum() == len(pts)
        q = pts[rng.integers(0, len(pts), 300)] + rng.normal(0, 0.2, (300, 4)).astype(np.float32)
        gp, gd, gc = g.Nearest_Search(q, 5)
        for i in range(len(q)):
            d = ((q[i, 0] - pts[:, 0]) ** 2 + (q[i, 1] - pts[:, 1]) ** 2) + (q[i, 2] - pts[:, 2]) ** 2
            assert np.array_equal(gd[i], np.sort(d)[:5])
    st = g.dir_stats()
    assert st["enabled"] and st["walked"] < 300 * 12                          # and the directory is still answering most queries
