"""CPU suite: the oracle's PoseOptimizationClient and OptimizeSim3 against runs where the REFERENCE'S OWN code does everything but the
6x6 / 7x7 Cholesky: g2o's Levenberg-Marquardt driver over g2o's VertexSE3Expmap / EdgeSE3ProjectXYZOnlyPose and VertexSim3Expmap /
EdgeSim3ProjectXYZ / EdgeInverseSim3ProjectXYZ with Huber kernels (oracle/ref_single_full_wrap.cpp -> oracle/_ref/libsingle_full_ref.so).
Estimates bit for bit, flags and counts exact.  The reference's outputs are stored under
tests/golden/reference (tests/reference_outputs.py)."""
import numpy as np
import pytest

from ccm_slam_b200 import synth
from tests.reference_outputs import Recorded, same


@pytest.fixture(scope="module")
def ref(oracle):
    return Recorded(oracle, __file__, oracle.ref_single_full)


def pose_args(d):
    return d["Tcw0"], d["Xw"], d["uv"], d["inv_sigma2"], d["intr"]


def sim3_args(d, fix):
    return d["S12_0"], d["P1c"], d["P2c"], d["uv1"], d["uv2"], d["w1"], d["w2"], d["K1"], d["K2"], d["th2"], fix


@pytest.mark.parametrize("n,seed,frac,noise", [(300, 11, 0.15, 0.8), (60, 12, 0.3, 0.8), (1000, 13, 0.05, 0.8), (12, 14, 0.0, 0.8), (400, 15, 0.5, 2.5),
                                                (9, 16, 0.2, 0.8), (3, 17, 0.0, 0.8), (2, 18, 0.0, 0.8)])
def test_pose_optimization(ref, n, seed, frac, noise):
    d = synth.make_pose_opt(n=n, seed=seed, outlier_frac=frac, noise_px=noise)
    T, out, nin = ref.pose_optimize(*pose_args(d)); Tr, outr, ninr = ref.ref_pose_optimize(*pose_args(d))
    assert nin == ninr and same(out, outr) and same(T, Tr)
    if n < 3:
        assert nin == 0 and same(T, d["Tcw0"])
    if frac >= 0.15 and n >= 60:
        assert 0 < out.sum() < n


def test_pose_optimization_bad_start(ref):
    """a start far enough that early rounds reject steps and flip many edges between inlier and outlier"""
    hit = 0
    for seed in range(30, 36):
        d = synth.make_pose_opt(n=150, seed=seed, outlier_frac=0.25, pose_noise=(0.15, 0.5))
        a = ref.pose_optimize(*pose_args(d)); b = ref.ref_pose_optimize(*pose_args(d))
        assert a[2] == b[2] and same(a[1], b[1]) and same(a[0], b[0])
        hit += a[1].sum() > 40
    assert hit >= 1


@pytest.mark.parametrize("n,seed,fix,frac", [(120, 12, False, 0.2), (120, 12, True, 0.2), (40, 21, False, 0.2), (80, 22, True, 0.0), (80, 23, False, 0.0),
                                             (12, 5, False, 0.6), (9, 6, False, 0.0), (200, 24, False, 0.4)])
def test_sim3_optimization(ref, n, seed, fix, frac):
    d = synth.make_sim3_opt(n=n, seed=seed, fix_scale=fix, outlier_frac=frac)
    S, inl, nin = ref.sim3_optimize(*sim3_args(d, fix)); Sr, inlr, ninr = ref.ref_sim3_optimize(*sim3_args(d, fix))
    assert nin == ninr and same(inl, inlr) and same(S, Sr)
    if n < 10:
        assert nin == 0 and same(S, d["S12_0"])        # fewer than 10 pairs survive: g2oS12 is left alone
    if fix and nin:
        assert S[7] == d["S12_0"][7]
