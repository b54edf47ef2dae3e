"""CPU suite: the oracle's Lie groups, edge errors, Jacobians (analytic and numeric), robust weighting and quadratic forms against the
REFERENCE'S OWN g2o types compiled in place (oracle/ref_g2o_wrap.cpp -> oracle/_ref/libg2o_types_ref.so): se3quat.h, sim3.h, se3_ops.hpp,
types_{sba,six_dof_expmap,seven_dof_expmap}.cpp, base_{vertex,edge,unary_edge,binary_edge}.h(pp), robust_kernel_impl.cpp.  Eigen itself is
absent; a stand-in (oracle/ref_stub/Eigen) supplies the small fixed-size arithmetic, eagerly and in index order, so everything below is
compared BIT FOR BIT: formulas, branch thresholds, expression grouping, float/double members, which Hessian block is written transposed.
Compiling the reference this way found four places where the oracle's restatement differed in the last bits or in a threshold (each
fixed in the oracle and noted there): RobustKernelHuber keeps delta^2 in a float; Sim3::log groups (B*Omega)*Omega; the point Jacobian
groups ((-1/z)*tmp)*R; the pose-landmark block is B^T(A^T Omega)^T without a kernel and (B^T wOmega)A with one; the unary edge's b is
((rho1 A^T) Omega) e.  The reference's outputs are stored under tests/golden/reference (tests/reference_outputs.py)."""
import numpy as np
import pytest

from ccm_slam_b200 import synth
from tests.reference_outputs import Recorded, same


@pytest.fixture(scope="module")
def sides(oracle):
    rec = Recorded(oracle, __file__, oracle.ref_g2o)
    return oracle.Pieces("oracle"), rec.obj("Pieces", lambda: oracle.Pieces("ref")), rec


def eq(a, b):
    return same(a, b)


def test_se3(sides):
    O, R, orc = sides
    rng = np.random.default_rng(0)
    n_small = 0
    for k in range(400):
        scale = [1e-9, 1e-6, 0.99e-5, 1.01e-5, 1e-3, 0.3, 2.0, 3.1][k % 8]      # both sides of the theta < 1e-5 quirk
        u = np.r_[rng.normal(0, 1, 3) * scale / np.sqrt(3), rng.normal(0, 2, 3)]
        n_small += np.linalg.norm(u[:3]) < 1e-5
        a = O.vec("se3_exp", 7, u)
        assert eq(a, R.vec("se3_exp", 7, u))
        b = O.vec("se3_exp", 7, rng.normal(0, 1, 6)); x = rng.normal(0, 3, 3)
        assert eq(O.vec("se3_mul", 7, a, b), R.vec("se3_mul", 7, a, b))      # includes normalizeRotation (w >= 0, then unit norm)
        assert eq(O.vec("se3_map", 3, a, x), R.vec("se3_map", 3, a, x))
        assert eq(R.vec("se3_mul", 7, R.vec("se3_exp", 7, u), b), orc.ref_vertex_oplus(0, b, u))   # VertexSE3Expmap::oplusImpl = exp(u) * T
    assert 50 < n_small < 350
    # Converter::toSE3Quat / toCvMat: float Tcw -> SE3Quat(R, t) -> float; all four branches of Quaterniond(Matrix3d)
    from scipy.spatial.transform import Rotation
    for rv in ([0.1, 0.2, -0.1], [3.0, 0.1, 0.1], [0.1, 3.0, 0.1], [0.1, 0.1, 3.0], [0, 0, 0], [2.2, -2.2, 0.3]):
        T = np.eye(4, dtype=np.float32)
        T[:3, :3] = Rotation.from_rotvec(rv).as_matrix().astype(np.float32); T[:3, 3] = np.float32([0.3, -1.2, 2.5])
        qt = orc.pose_from_Tcw_f32(T)
        assert eq(qt, R.vec("se3_from_Rt", 7, T[:3, :3].astype(np.float64).ravel(), T[:3, 3].astype(np.float64)))
        to_f32 = lambda q: R.live.vec("se3_homogeneous", 16, q).astype(np.float32).reshape(4, 4)
        assert eq(orc.pose_to_Tcw_f32(qt), orc.call("se3_homogeneous_f32", to_f32, qt))


def test_sim3(sides):
    O, R, orc = sides
    rng = np.random.default_rng(1)
    branches = set()
    for k in range(600):
        th = [1e-9, 0.99e-5, 1.01e-5, 0.02, 0.7, 3.0][k % 6]; sg = [0.0, 0.99e-5, -0.99e-5, 1.01e-5, -0.3, 0.8][(k // 6) % 6]
        u = np.r_[rng.normal(0, 1, 3) * th / np.sqrt(3), rng.normal(0, 2, 3), sg]
        branches.add((np.linalg.norm(u[:3]) < 1e-5, abs(sg) < 1e-5))
        s = O.vec("sim3_exp", 8, u)
        assert eq(s, R.vec("sim3_exp", 8, u))
        assert eq(O.vec("sim3_log", 7, s), R.vec("sim3_log", 7, s))            # incl. (B*Omega)*Omega and the 3x3 partial-pivot solve
        assert eq(O.vec("sim3_inv", 8, s), R.vec("sim3_inv", 8, s))
        t = O.vec("sim3_exp", 8, rng.normal(0, 0.6, 7)); x = rng.normal(0, 3, 3)
        assert eq(O.vec("sim3_mul", 8, s, t), R.vec("sim3_mul", 8, s, t))
        assert eq(O.vec("sim3_map", 3, s, x), R.vec("sim3_map", 3, s, x))
        for fix in (0, 1):                                                       # VertexSim3Expmap::oplusImpl, _fix_scale zeroes the 7th
            v = u.copy(); v[6] = 0 if fix else v[6]
            assert eq(O.vec("sim3_mul", 8, O.vec("sim3_exp", 8, v), t), orc.ref_vertex_oplus(1, t, u, fix))
    assert len(branches) == 4
    # log near the identity rotation (d > 1 - eps) with and without scale
    for sg in (0.0, 0.4):
        s = O.vec("sim3_exp", 8, np.r_[1e-7, -2e-7, 1e-7, 0.5, 0.1, -0.2, sg])
        assert eq(O.vec("sim3_log", 7, s), R.vec("sim3_log", 7, s))
    assert eq(orc.ref_vertex_oplus(2, [1.0, 2.0, 3.0], [0.5, -0.25, 1e-9]), np.array([1.5, 1.75, 3.0 + 1e-9]))


def test_huber_float_square(sides):
    O, R, _ = sides
    for d in (float(np.float32(np.sqrt(5.99))), float(np.float32(np.sqrt(5.991))), np.sqrt(5.99), 1.0, float(np.float32(np.sqrt(10.0)))):
        d2f = float(np.float32(d * d))
        for e in (0.0, 0.3, d2f, np.nextafter(d2f, 0), np.nextafter(d2f, 100), d * d, np.nextafter(d * d, 100), 7.0, 1e3, 1e8):
            assert eq(O.huber(e, d), R.huber(e, d)), (d, e)
    d = float(np.float32(np.sqrt(5.99)))
    assert float(np.float32(d * d)) != d * d and R.huber(float(np.float32(d * d)), d)[2] == 0      # the rounded square is the threshold


@pytest.mark.parametrize("name", ["tiny", "small", "cfg2"])
def test_ba_edges_and_quadratic_form(sides, name):
    """EdgeSE3ProjectXYZ::computeError / linearizeOplus / chi2, Huber, and BaseBinaryEdge::constructQuadraticForm accumulated over a whole
    problem in edge order into mapped Hpp / Hll / Hpl blocks, as BlockSolver::buildSystem drives them."""
    O, R, _ = sides
    p = synth.make_config(name) if name != "cfg2" else synth.make_config("cfg2", P=500)
    for robust, delta in ((True, np.sqrt(5.99)), (True, float(np.float32(np.sqrt(5.991)))), (False, 1.0)):
        a = O.ba_linearize(p, robust=robust, huber_delta=delta); b = R.ba_linearize(p, robust=robust, huber_delta=delta)
        for k in a:
            assert eq(a[k], b[k]), k
        if robust:
            assert (a["rho1"] < 1).sum() > 5 and (a["rho1"] == 1).sum() > 5
        a = O.ba_build(p, robust=robust, huber_delta=delta); b = R.ba_build(p, robust=robust, huber_delta=delta)
        for k in a:
            assert eq(a[k], b[k]), k
        assert np.abs(a["W"]).max() > 0 and (np.abs(a["Hpp"][p.fixed != 0]).max() == 0 if (p.fixed != 0).any() else True)
    # second-round flags of LocalBundleAdjustmentClient: level-1 edges are left out, kernels dropped on the rest
    rng = np.random.default_rng(2)
    p2 = p.copy(); p2.edge_flags = (rng.random(p.E) < 0.2).astype(np.uint8) | 2
    a = O.ba_build(p2); b = R.ba_build(p2)
    for k in a:
        assert eq(a[k], b[k]), k


def test_pose_only_edges(sides):
    """EdgeSE3ProjectXYZOnlyPose (BaseUnaryEdge): error, analytic Jacobian with invz, and the unary-edge quadratic form."""
    O, R, _ = sides
    for seed in (11, 12, 13):
        pp = synth.make_pose_opt(n=200, seed=seed)
        for robust in (1, 0):
            args = (pp["Tcw0"], pp["Xw"], pp["uv"], pp["inv_sigma2"], pp["intr"], robust, float(np.float32(np.sqrt(5.991))))
            for x, y in zip(O.pose_opt_build(*args), R.pose_opt_build(*args)):
                assert eq(x, y)


def test_sim3_projection_edges(sides):
    """EdgeSim3ProjectXYZ / EdgeInverseSim3ProjectXYZ with a fixed point vertex: errors through cam_map1 / cam_map2, the numeric Jacobian of
    BaseBinaryEdge::linearizeOplus (delta 1e-9, push / oplus / pop on the Sim3 vertex, _fix_scale), robust quadratic form."""
    O, R, _ = sides
    for seed in (12, 13):
        sp = synth.make_sim3_opt(n=100, seed=seed)
        for fix in (0, 1):
            for robust in (1, 0):
                args = (sp["S12_0"], sp["P1c"], sp["P2c"], sp["uv1"], sp["uv2"], sp["w1"], sp["w2"], sp["K1"], sp["K2"], fix, robust,
                        float(np.float32(np.sqrt(sp["th2"]))))
                a = O.sim3_opt_build(*args); b = R.sim3_opt_build(*args)
                for x, y in zip(a, b):
                    assert eq(x, y)
                if fix:
                    assert np.all(a[0][6] == 0) and np.all(a[0][:, 6] == 0) and a[1][6] == 0      # a frozen scale has no curvature


def test_essential_graph_edge(sides):
    """EdgeSim3::computeError = log(C * Si * Sj^-1) and its numeric Jacobians with respect to both vertices."""
    O, R, _ = sides
    rng = np.random.default_rng(3)
    for k in range(60):
        si, sj = [O.vec("sim3_exp", 8, rng.normal(0, 0.5, 7)) for _ in range(2)]
        # a measurement near Sj * Si^-1 (small residual, as in a converging graph) or far from it
        c = O.vec("sim3_mul", 8, sj, O.vec("sim3_inv", 8, si))
        if k % 2:
            c = O.vec("sim3_mul", 8, O.vec("sim3_exp", 8, rng.normal(0, 0.02, 7)), c)
        else:
            c = O.vec("sim3_exp", 8, rng.normal(0, 0.5, 7))
        assert eq(O.vec("pgo_edge_error", 7, c, si, sj), R.vec("pgo_edge_error", 7, c, si, sj))
        for fix in (0, 1):
            a = O.pgo_edge_jacobian(c, si, sj, fix); b = R.pgo_edge_jacobian(c, si, sj, fix)
            assert eq(a[0], b[0]) and eq(a[1], b[1])
            if fix:
                assert np.all(a[0][:, 6] == 0) and np.all(a[1][:, 6] == 0)
