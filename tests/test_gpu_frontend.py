"""Scan front end on the GPU (SURVEY.md §8f rows 3-4) against the CPU oracle: de-skew (UndistortPcl backward pass),
pcl::VoxelGrid down-sampling, and the device-resident chain raw -> de-skew -> down-sample -> update."""
import numpy as np
import pytest

from fast_lio_b200 import api, synth
from oracle import bind
from reference_tape import ReferenceTree

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tree(problems):
    pr = problems("small")
    t = api.KdTree(0, 0.5)
    t.Build(pr.map_pts)
    return t


@pytest.fixture(scope="module")
def raw(problems):
    pr = problems("small")
    return synth.make_raw_scan(pr.scene, 40_000, pr.x_true, seed=21)


def _ulps(a, b):
    a = np.asarray(a, np.float32); b = np.asarray(b, np.float32)
    return np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.spacing(np.maximum(np.abs(a), np.abs(b)).astype(np.float32)).astype(np.float64)


def test_undistort_matches_oracle(tree, raw):
    s = api.Scan(tree)
    s.upload(raw.xyzi, raw.offset_ms)
    s.undistort(raw.imu_pose, raw.x_end)
    got = s.download(0)
    want, ts = bind.undistort(raw.xyzi, raw.offset_ms, raw.imu_pose, raw.x_end)
    assert got.shape == want.shape
    assert np.array_equal(got[:, 3], want[:, 3])                      # same (stable) time order, intensity untouched
    # FP64 on both sides, results rounded to float32: device sin/cos differ from glibc in the last bit of a double,
    # which moves a float32 result by at most one ulp, rarely
    u = _ulps(got[:, :3], want[:, :3])
    assert u.max() <= 1.0
    assert (u > 0).mean() < 1e-3
    order = np.argsort(raw.offset_ms, kind="stable")
    assert np.abs(got[1:, :3] - raw.truth_end[order][1:]).max() < 5e-6   # and it does undo the motion


def test_undistort_quirks_match_oracle(tree, raw):
    """Negative IMU offsets (samples before the first point) and the re-compensated first point (IMU_Processing.hpp:343)."""
    poses = np.vstack([raw.imu_pose[:1], raw.imu_pose[:1], raw.imu_pose[1:]])
    poses[1, 0] = -0.004
    t = raw.offset_ms.copy()
    t[np.argmin(t)] = 7.0                                             # no point at offset 0: the earliest one is at 7 ms... or later
    s = api.Scan(tree)
    s.upload(raw.xyzi, t)
    s.undistort(poses, raw.x_end)
    got = s.download(0)
    want, _ = bind.undistort(raw.xyzi, t, poses, raw.x_end)
    assert _ulps(got[:, :3], want[:, :3]).max() <= 1.0
    # fewer than two poses: only the sort happens
    s.upload(raw.xyzi, raw.offset_ms)
    s.undistort(raw.imu_pose[:1], raw.x_end)
    assert np.array_equal(s.download(0), raw.xyzi[np.argsort(raw.offset_ms, kind="stable")])


@pytest.mark.parametrize("leaf", [0.5, 0.25])
def test_voxelgrid_bit_exact(tree, raw, leaf):
    s = api.Scan(tree)
    s.upload(raw.xyzi, raw.offset_ms)
    n = s.voxel_downsample(leaf)
    got = s.download(1)
    want = bind.voxelgrid(raw.xyzi, leaf)
    assert n == len(want) == len(got)
    assert np.array_equal(got, want)                                  # float32 sums in the same order: bit-exact, same cell order


def test_voxelgrid_edge_cases(tree):
    s = api.Scan(tree)
    s.upload(np.zeros((0, 4), np.float32), np.zeros(0, np.float32))
    assert s.voxel_downsample(0.5) == 0 and len(s.download(1)) == 0
    one = np.array([[1.25, -3.5, 0.75, 9.0]], np.float32)
    s.upload(one, np.zeros(1, np.float32))
    assert s.voxel_downsample(0.5) == 1 and np.array_equal(s.download(1), one)
    rng = np.random.default_rng(0)
    cloud = np.c_[rng.uniform(-0.24, 0.24, (500, 3)) + 0.25, rng.uniform(0, 255, 500)].astype(np.float32)   # 500 points, one cell
    s.upload(cloud, np.zeros(500, np.float32))
    assert s.voxel_downsample(0.5) == 1
    assert np.array_equal(s.download(1), bind.voxelgrid(cloud, 0.5))
    far = np.array([[0, 0, 0, 1.0], [300, 300, 300, 2.0], [1, 1, 1, 3.0]], np.float32)
    s.upload(far, np.zeros(3, np.float32))
    assert s.voxel_downsample(0.1) == 3 and np.array_equal(s.download(1), far)    # PCL's leaf-too-small exit: output = input
    with pytest.raises(api.FastLioError):
        s.voxel_downsample(0.0)


def test_resident_chain_matches_host_chain(problems, tree, raw):
    """raw -> de-skew -> voxel grid -> update, all in HBM, equals the same update fed with the down-sampled cloud from
    the host, and tracks the CPU oracle run on the oracle's own front end."""
    pr = problems("small")
    f = api.Esekf(tree, max_points=50_000, max_iter=3)
    s = api.Scan(tree)
    s.upload(raw.xyzi, raw.offset_ms)
    s.undistort(raw.imu_pose, raw.x_end)
    n = s.voxel_downsample(0.5)
    assert 1000 < n < len(raw.xyzi)
    x_dev, P_dev, _ = s.update(f, pr.x_prior, pr.P_prior, pr.R)
    down = s.download(1)
    x_host, P_host, _ = f.update_iterated_dyn_share_modified(down, pr.x_prior, pr.P_prior, pr.R)
    assert np.array_equal(x_dev, x_host) and np.array_equal(P_dev, P_host)
    # the oracle's chain (its own de-skew + voxel grid + update on the reference ikd-Tree / the port)
    o_pts, _ = bind.undistort(raw.xyzi, raw.offset_ms, raw.imu_pose, raw.x_end)
    o_down = bind.voxelgrid(o_pts, 0.5)
    assert len(o_down) == n
    ot = bind.KdTree(pr.map_pts, "auto")
    r = bind.update_iterated(ot, o_down, pr.x_prior, pr.P_prior, 3, pr.R)
    assert np.abs(x_dev[:3] - r.x[:3]).max() < 1e-4                   # north-star tolerance: 1e-4 m / 1e-4 rad
    assert np.abs(x_dev[3:7] - r.x[3:7]).max() < 1e-4
    assert np.abs(x_dev - r.x).max() < 1e-4
    # map_incremental runs off the same resident cloud
    n_add, n_no, added = f.map_incremental(0.5, True)
    assert n_add + n_no > 0 and added >= 0


def test_localmap_segment_deletes_from_the_map(problems):
    pr = problems("small")
    g = api.KdTree(0, 0.5); g.Build(pr.map_pts)
    ours = api.LocalMap(40.0, 8.0)
    ref = bind.LocalMap(40.0, 8.0)
    rt = ReferenceTree("localmap_segment", pr.map_pts)
    pos = np.array(pr.x_true[:3], dtype=np.float64)
    total = 0
    for k in range(12):
        pos = pos + np.array([1.5, 0.7, 0.0])
        boxes, n_deleted = ours.segment(pos, g)
        b_ref = ref.segment(pos)
        assert np.array_equal(boxes, b_ref)
        if len(b_ref):
            assert n_deleted == rt.delete_boxes(b_ref)
            assert g.validnum() == rt.validnum()
        total += n_deleted
    assert total > 0
