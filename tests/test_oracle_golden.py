"""CPU: the oracle against the committed golden vectors (tests/golden/*.npz, minted by
tests/golden/make_golden.py from the reference's own ikd-Tree + the restatement) and against
independent numpy formulations of its pieces."""
import os

import numpy as np
import pytest

from fast_lio_b200 import synth
from oracle import bind
from reference_tape import ReferenceTree

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def world_queries(pr):
    q = np.zeros((len(pr.scan), 4), dtype=np.float32)
    tmp = np.zeros(3, dtype=np.float32)
    for i in range(len(pr.scan)):
        bind.lib().oracle_transform_point(pr.x_prior, np.ascontiguousarray(pr.scan[i, :3]), tmp)
        q[i, :3] = tmp
    return q


@pytest.mark.parametrize("name", ["tiny", "small"])
def test_generator_is_stable(problems, name):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    pr = problems(name)
    assert float(pr.map_pts.astype(np.float64).sum()) == float(g["map_sum"])
    assert float(pr.scan.astype(np.float64).sum()) == float(g["scan_sum"])
    assert np.array_equal(pr.x_prior, g["x_prior"])


@pytest.mark.parametrize("name", ["tiny", "small"])
@pytest.mark.parametrize("backend", ["port", "reference"])
def test_knn_golden(problems, name, backend):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    pr = problems(name)
    t = ReferenceTree(f"knn_{name}", pr.map_pts) if backend == "reference" else bind.KdTree(pr.map_pts, backend)
    p, d, c = t.knn(world_queries(pr), 5)
    assert np.array_equal(c, g["knn_cnt"]) and np.array_equal(d, g["knn_d2"]) and np.array_equal(p, g["knn_pts"])


@pytest.mark.parametrize("name", ["tiny", "small"])
@pytest.mark.parametrize("extr", [0, 1])
def test_update_golden(problems, name, extr):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    pr = problems(name)
    t = bind.KdTree(pr.map_pts, "port")
    o = bind.update_iterated(t, pr.scan, pr.x_prior, pr.P_prior, pr.cfg.max_iter, pr.R, pr.limit, extr, nthreads=2)
    assert np.array_equal(np.array([p["effct"] for p in o.passes]), g[f"effct_{extr}"])
    assert np.array_equal(np.array([p["searched"] for p in o.passes]), g[f"searched_{extr}"])
    assert np.array_equal(np.array([p["converged"] for p in o.passes]), g[f"converged_{extr}"])
    assert np.allclose(np.stack([p["HtH"] for p in o.passes]), g[f"HtH_{extr}"], rtol=1e-12, atol=1e-9)
    assert np.allclose(o.x, g[f"x_{extr}"], rtol=0, atol=1e-12)
    assert np.allclose(o.P, g[f"P_{extr}"], rtol=1e-9, atol=1e-15)
    assert np.array_equal(o.selected, g[f"selected_{extr}"])


def test_update_reduces_error(problems):
    pr = problems("small")
    t = bind.KdTree(pr.map_pts, "port")
    o = bind.update_iterated(t, pr.scan, pr.x_prior, pr.P_prior, pr.cfg.max_iter, pr.R, pr.limit, 0)
    assert np.abs(pr.x_prior[:3] - pr.x_true[:3]).max() > 0.02
    assert np.abs(o.x[:3] - pr.x_true[:3]).max() < 5e-3
    assert (np.diag(o.P)[:6] < np.diag(pr.P_prior)[:6]).all()
    assert np.allclose(o.P, o.P.T, atol=1e-12)


def test_esti_plane_against_lstsq():
    """esti_plane (float32 column-pivoted QR) vs float64 least squares on well-conditioned planes."""
    rng = np.random.default_rng(0)
    for _ in range(200):
        n = rng.normal(size=3); n /= np.linalg.norm(n)
        d = rng.uniform(1.0, 5.0)
        c = -d * n + rng.normal(size=3) * 0.0
        u = np.cross(n, [1, 0, 0]); u /= np.linalg.norm(u); v = np.cross(n, u)
        pts = np.array([c + rng.uniform(-1, 1) * u + rng.uniform(-1, 1) * v + rng.normal(0, 0.002) * n for _ in range(5)], dtype=np.float32)
        ok, pabcd = bind.esti_plane(pts, 0.1)
        sol, *_ = np.linalg.lstsq(pts.astype(np.float64), -np.ones(5), rcond=None)
        nn = np.linalg.norm(sol)
        ref = np.array([*(sol / nn), 1.0 / nn])
        assert ok
        assert np.allclose(pabcd, ref, atol=5e-4)
    # points far off a plane are rejected
    ok, _ = bind.esti_plane(np.array([[0, 0, 1], [1, 0, 1.5], [0, 1, 0.5], [1, 1, 1.9], [2, 2, 1]], dtype=np.float32), 0.1)
    assert not ok


def test_manifold_roundtrip():
    """x [+] (y [-] x) == y for the compound state (boxplus/boxminus of vect, SO3, S2)."""
    rng = np.random.default_rng(1)
    L = bind.lib()
    x = synth.true_state("avia")
    for _ in range(50):
        d = rng.normal(0, 0.02, 23)
        y = x.copy()
        L.oracle_state_boxplus(y, d)
        back = np.zeros(23)
        L.oracle_state_boxminus(y, x, back)
        assert np.allclose(back, d, atol=1e-9)
        assert abs(np.linalg.norm(y[23:26]) - synth.G_LEN) < 1e-9
        assert abs(np.linalg.norm(y[3:7]) - 1.0) < 1e-3


def test_inverse_matches_numpy():
    rng = np.random.default_rng(2)
    A = rng.normal(size=(23, 23)); A = A @ A.T + 23 * np.eye(23)
    out = np.zeros((23, 23))
    assert bind.lib().oracle_inverse(np.ascontiguousarray(A), out, 23) == 0
    assert np.allclose(out, np.linalg.inv(A), rtol=1e-10, atol=1e-13)


def test_A_matrix_matches_series():
    L = bind.lib()
    v = np.array([0.03, -0.02, 0.05])
    out = np.zeros(9)
    L.oracle_A_matrix(v, out)
    K = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    n = np.linalg.norm(v)
    ref = np.eye(3) + (1 - np.cos(n)) / n**2 * K + (1 - np.sin(n) / n) / n**2 * K @ K
    assert np.allclose(out.reshape(3, 3), ref, atol=1e-14)


def test_A_matrix_is_the_left_jacobian_of_exp():
    """Independent of the closed form: Exp(v + dv) ~= Exp(A(v) dv) Exp(v) to first order (scipy's rotation vectors)."""
    from scipy.spatial.transform import Rotation as Rot
    L = bind.lib()
    rng = np.random.default_rng(5)
    for _ in range(20):
        v = rng.normal(0, 0.3, 3)
        A = np.zeros(9); L.oracle_A_matrix(v, A); A = A.reshape(3, 3)
        J = np.zeros((3, 3))
        eps = 1e-6
        for a in range(3):
            dv = np.zeros(3); dv[a] = eps
            J[:, a] = (Rot.from_rotvec(v + dv) * Rot.from_rotvec(v).inv()).as_rotvec() / eps
        assert np.allclose(A, J, atol=5e-6)


def test_boxplus_is_right_multiplication_by_exp():
    """SO3 [+] (SOn.hpp:233-236): q [+] d = q * Exp(d); checked against scipy, for rot and offset_R_L_I; vectors add;
    the S2 gravity keeps its length and moves by ~|d| on the sphere."""
    from scipy.spatial.transform import Rotation as Rot
    L = bind.lib()
    rng = np.random.default_rng(6)
    x = synth.true_state("velodyne")
    for _ in range(20):
        d = rng.normal(0, 0.05, 23)
        y = x.copy(); L.oracle_state_boxplus(y, d)
        for xo, do in ((3, 3), (7, 6)):
            want = (Rot.from_quat(x[xo:xo + 4]) * Rot.from_rotvec(d[do:do + 3])).as_quat()
            got = y[xo:xo + 4] / np.linalg.norm(y[xo:xo + 4])
            assert min(np.abs(got - want).max(), np.abs(got + want).max()) < 1e-12
        assert np.allclose(y[0:3], x[0:3] + d[0:3]) and np.allclose(y[14:17], x[14:17] + d[12:15])
        ang = np.arccos(np.clip(np.dot(y[23:26], x[23:26]) / synth.G_LEN ** 2, -1, 1))
        assert abs(ang - np.linalg.norm(d[21:23])) < 1e-3 * max(1.0, np.linalg.norm(d[21:23]) * 1e3)


def test_first_pass_equals_the_closed_form_kalman_step(problems):
    """With x = x_propagated (first pass) every manifold Jacobian is the identity and the pass is a plain Kalman step:
    dx = (H^T H / R + P^-1)^-1 H^T z / R on the 12 observed DOF (esekfom.hpp:1784-1817).  Recompute it with numpy from
    the oracle's own H^T H / H^T h of that pass and compare the state it reports after the pass."""
    pr = problems("small")
    t = bind.KdTree(pr.map_pts, "port")
    o = bind.update_iterated(t, pr.scan, pr.x_prior, pr.P_prior, pr.cfg.max_iter, pr.R, pr.limit, 0)
    p0 = o.passes[0]
    HtH = np.zeros((23, 23)); HtH[:12, :12] = p0["HtH"]
    Hth = np.zeros(23); Hth[:12] = p0["Hth"]
    # the model: z = -h (laserMapping.cpp:751 stores h = -pd2), measurement noise R I
    dx = np.linalg.solve(HtH / pr.R + np.linalg.inv(pr.P_prior), Hth / pr.R)
    want = pr.x_prior.copy()
    bind.lib().oracle_state_boxplus(want, np.ascontiguousarray(dx))
    assert np.abs(want - p0["x_after"]).max() < 1e-9


@pytest.mark.parametrize("extr", [0, 1])
def test_update_lands_on_the_map_estimate(problems, extr):
    """An iterated EKF update is Gauss-Newton on  |x [-] x_prior|^2_{P^-1} + sum z_i(x)^2 / R  (FAST-LIO2 eq. 17-20): with the
    correspondences and planes of the last search pass held fixed, the state the oracle returns must be a stationary point
    of that cost.  The cost and its gradient are evaluated here with numpy and central differences -- nothing of the
    update's own Jacobian code is reused -- so a wrong Jacobian row, congruence block or sign would leave a gradient."""
    pr = problems("small")
    t = bind.KdTree(pr.map_pts, "port")
    L = bind.lib()
    o = bind.update_iterated(t, pr.scan, pr.x_prior, pr.P_prior, pr.cfg.max_iter, pr.R, pr.limit, extr)
    sel = o.selected.astype(bool)
    assert sel.sum() > 500
    planes = np.zeros((len(pr.scan), 4))
    for i in np.flatnonzero(sel):
        ok, pl = bind.esti_plane(o.nearest[i, :, :3], 0.1)
        assert ok
        planes[i] = pl
    Pinv = np.linalg.inv(pr.P_prior)
    pts = pr.scan[sel, :3].astype(np.float64)
    pl = planes[sel]

    def cost(x):
        r = np.zeros(23)
        L.oracle_state_boxminus(np.ascontiguousarray(x), pr.x_prior, r)
        R = synth.quat_to_mat(x[3:7]); Rl = synth.quat_to_mat(x[7:11])
        pw = (pts @ Rl.T + x[11:14]) @ R.T + x[0:3]
        z = (pw * pl[:, :3]).sum(axis=1) + pl[:, 3]
        return r @ Pinv @ r + (z * z).sum() / pr.R

    def grad(x0):
        g = np.zeros(23)
        for a in range(23):
            d = np.zeros(23); d[a] = 1e-6
            xp = x0.copy(); L.oracle_state_boxplus(xp, d)
            xm = x0.copy(); L.oracle_state_boxplus(xm, -d)
            g[a] = (cost(xp) - cost(xm)) / 2e-6
        return g

    g_prior, g_post = grad(pr.x_prior), grad(o.x)
    assert cost(o.x) < 0.1 * cost(pr.x_prior)
    assert np.linalg.norm(g_post) < 1e-5 * np.linalg.norm(g_prior)


@pytest.mark.parametrize("extr", [0, 1])
def test_posterior_covariance_is_the_inverse_information(problems, extr):
    """esekfom.hpp:1834-1927 assembles P = L - K_x P with the manifold congruences; for the small corrections of a scan
    (|dx| ~ 1e-2) those are the identity to first order, so P must equal (P_prior^-1 + H^T H / R)^-1 with the H^T H of the
    last pass -- computed here with numpy from the oracle's own normal equations."""
    pr = problems("small")
    t = bind.KdTree(pr.map_pts, "port")
    o = bind.update_iterated(t, pr.scan, pr.x_prior, pr.P_prior, pr.cfg.max_iter, pr.R, pr.limit, extr)
    HtH = np.zeros((23, 23)); HtH[:12, :12] = o.passes[-1]["HtH"]
    want = np.linalg.inv(np.linalg.inv(pr.P_prior) + HtH / pr.R)
    scale = np.sqrt(np.outer(np.diag(want), np.diag(want)))
    assert (np.abs(o.P - want) / scale).max() < 1e-4
    # the reference never symmetrises P; with extrinsic estimation the barely observable LiDAR-IMU rotation leaves 1e-5-level asymmetry
    assert (np.abs(o.P - o.P.T) / scale).max() < 1e-4 and np.linalg.eigvalsh(0.5 * (o.P + o.P.T)).min() > 0
