"""CPU suite: the oracle's essential-graph optimisation against a run where the REFERENCE'S OWN code does everything but the sparse
factorisation: g2o's Levenberg-Marquardt driver over g2o's VertexSim3Expmap / EdgeSim3 — Sim3::log errors, the numeric Jacobians of
BaseBinaryEdge::linearizeOplus, constructQuadraticForm into upper-triangle 7x7 blocks with the transposed write, oplus with _fix_scale
(oracle/ref_pgo_full_wrap.cpp -> oracle/_ref/libpgo_full_ref.so).  Traces and final vertices bit for bit.  The reference's outputs are stored under
tests/golden/reference (tests/reference_outputs.py)."""
import numpy as np
import pytest

from ccm_slam_b200 import synth
from tests.reference_outputs import Recorded
from tests.reference_outputs import same as same_array


class _Side:
    def __init__(self, oracle, level):
        self.pgo_solve = oracle.pgo_solve
        self.ref_pgo_solve = oracle.ref_pgo_solve if level == "full" else oracle.ref_pgo_block_solve


# "full": the reference's LM driver, vertices and edges; "block": plus its BlockSolver_7_3 (block allocation, buildSystem, damping,
# the non-Schur solve) — only LinearSolver::solve, the sparse LDL^T, is the oracle's (oracle/ref_pgo_block_wrap.cpp)
@pytest.fixture(scope="module", params=["full", "block"])
def ref(oracle, request):
    live = oracle.ref_pgo_full if request.param == "full" else oracle.ref_pgo_block
    return _Side(Recorded(oracle, __file__, live, keep={"trace"}), request.param)


def same(a, b):
    assert a["iters_done"] == b["iters_done"] and len(a["trace"]) == len(b["trace"])
    for c in (0, 1, 2, 4, 5):
        if c == 1 and np.isnan(b["trace"][:, 1]).all():
            continue                # inside the reference's own BlockSolver the last trial's lambda is not visible
        assert same_array(a["trace"][:, c], b["trace"][:, c]), c
    assert a["chi2_initial"] == b["chi2_initial"] and a["chi2_final"] == b["chi2_final"] and a["lambda_final"] == b["lambda_final"]
    assert same_array(a["sim3"], b["sim3"])


@pytest.mark.parametrize("fix_scale", [False, True])
@pytest.mark.parametrize("K,n_loop,drift", [(60, 6, (0.002, 0.01, 0.002)), (200, 10, (0.005, 0.03, 0.004)), (40, 2, (0.02, 0.1, 0.01))])
def test_essential_graph_runs(ref, K, n_loop, drift, fix_scale):
    p = synth.make_pgo(K=K, n_loop=n_loop, fix_scale=fix_scale, drift=drift)
    seen_reject = False
    for lam in (1e-16, -1.0, 1e-3):       # Optimizer.cpp sets 1e-16; the computed and a moderate start exercise other trial patterns
        a = ref.pgo_solve(p, iterations=20, lambda_init=lam); b = ref.ref_pgo_solve(p, iterations=20, lambda_init=lam)
        same(a, b)
        assert a["chi2_final"] <= a["chi2_initial"]
        seen_reject |= bool((a["trace"][:, 4] > 1).any())
    if not fix_scale:
        assert seen_reject               # free scale: rejected trials (nu doubling) and the 10-trial stop occur


def test_fixed_vertices_stop_flag_and_empty(ref):
    p = synth.make_pgo(K=50, n_loop=4)
    rng = np.random.default_rng(1)
    p.fixed = (rng.random(50) < 0.3).astype(np.uint8); p.fixed[0] = 1         # edges with one fixed end, and some with both (left out)
    same(ref.pgo_solve(p, iterations=10, lambda_init=-1.0), ref.ref_pgo_solve(p, iterations=10, lambda_init=-1.0))
    stop = np.ones(1, np.uint8)
    same(ref.pgo_solve(p, iterations=10, stop=stop), ref.ref_pgo_solve(p, iterations=10, stop=stop))
    same(ref.pgo_solve(p, iterations=0), ref.ref_pgo_solve(p, iterations=0))
    p.fixed[:] = 1
    a = ref.pgo_solve(p, iterations=5); b = ref.ref_pgo_solve(p, iterations=5)
    assert a["iters_done"] == b["iters_done"] == -1 and same_array(a["sim3"], b["sim3"])
