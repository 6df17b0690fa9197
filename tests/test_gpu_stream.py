"""BASELINE config 4 in miniature: a stream of scans with Delete_Point_Boxes (window move),
update, map_incremental + Add_Points every scan -- device pipeline vs the CPU reference pipeline."""
import numpy as np
import pytest

from fast_lio_b200 import api, synth
from reference_tape import ReferenceTree
from semantics import map_incremental, sort_rows

pytestmark = pytest.mark.gpu


def test_map_incremental_matches_reference(problems):
    pr = problems("small")
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    f = api.Esekf(g, max_points=len(pr.scan), max_iter=pr.cfg.max_iter)
    x, P, _ = f.update_iterated_dyn_share_modified(pr.scan, pr.x_prior, pr.P_prior, pr.R)
    near, cnt = f.nearest(len(pr.scan))
    n_add, n_no, added = f.map_incremental(0.5, True)
    # CPU reference pipeline from the same update result
    r = ReferenceTree("map_incremental_small", pr.map_pts, downsample=0.5)      # fed the device's points: new bits need a new tape
    to_add, no_need = map_incremental(pr.scan, x, near, cnt, 0.5, True)
    assert (n_add, n_no) == (len(to_add), len(no_need))
    assert added == r.add(to_add, True)
    r.add(no_need, False)
    assert g.validnum() == r.validnum()
    assert np.array_equal(sort_rows(g.flatten()), sort_rows(r.flatten()))


def test_stream_of_scans(problems):
    """5 scans: the sensor advances 0.1 m per scan; state and map of the device pipeline track the CPU pipeline."""
    pr = problems("small")
    scene = pr.scene
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    f = api.Esekf(g, max_points=2000, max_iter=3)
    r = ReferenceTree("stream_of_scans_small", pr.map_pts, downsample=0.5)
    x_g = pr.x_prior.copy(); x_c = pr.x_prior.copy()
    P_g = pr.P_prior.copy(); P_c = pr.P_prior.copy()
    for step in range(5):
        xt = synth.true_state(pr.cfg.lidar, step)
        scan = synth.make_scan(scene, 800, xt, seed=100 + step)
        if step == 2:       # the local-map window moves: drop a slab (lasermap_fov_segment :257-270)
            box = np.array([[-1000, -1000, -1000, -60.0, 1000, 1000]], dtype=np.float32)
            assert g.Delete_Point_Boxes(box) == r.delete_boxes(box)
        # crude prediction: carry the state over, inflate the covariance
        P_g = P_g + np.eye(23) * 1e-4; P_c = P_c + np.eye(23) * 1e-4
        x_g, P_g, _ = f.update_iterated_dyn_share_modified(scan, x_g, P_g, pr.R)
        o = r.update_iterated(scan, x_c, P_c, 3, pr.R, pr.limit, 0)
        x_c, P_c = o.x, o.P
        assert np.abs(x_g[:3] - x_c[:3]).max() <= 1e-4 and np.abs(x_g[3:7] - x_c[3:7]).max() <= 1e-4
        n_add, n_no, added = f.map_incremental(0.5, True)
        to_add, no_need = map_incremental(scan, x_c, o.nearest, o.nearest_cnt, 0.5, True)
        assert (n_add, n_no) == (len(to_add), len(no_need))
        assert added == r.add(to_add, True)
        r.add(no_need, False)
        assert g.validnum() == r.validnum()
    assert np.array_equal(sort_rows(g.flatten()), sort_rows(r.flatten()))
    assert np.abs(x_g[:3] - synth.true_state(pr.cfg.lidar, 4)[:3]).max() < 0.02
