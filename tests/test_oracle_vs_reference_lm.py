"""CPU suite: the oracle's Levenberg-Marquardt control flow (SURVEY.md §8 row a8) against the REFERENCE'S OWN compiled
OptimizationAlgorithmLevenberg::solve (oracle/ref_lm_wrap.cpp: g2o's three optimization_algorithm*.cpp files compiled in place over
stand-in SparseOptimizer / Solver classes whose bodies are the oracle's linear algebra).  Both drivers run the same arithmetic, so
lambda, chi2, trial counts, iteration counts and the final state must agree to the last bit; anything else is a control-flow
difference.  The reference's outputs are stored under tests/golden/reference (tests/reference_outputs.py)."""
import numpy as np
import pytest

from ccm_slam_b200 import synth
from tests.reference_outputs import Recorded, same


class _Side:
    """the oracle's ba_solve next to one of the two reference-driven runs"""

    def __init__(self, oracle, driver):
        self.ba_solve = oracle.ba_solve
        self.ref_ba_solve = {"lm": oracle.ref_ba_solve, "full": oracle.ref_ba_full_solve, "block": oracle.ref_ba_block_solve}[driver]
        self.driver = driver


# "lm":   g2o's Levenberg-Marquardt driver over the oracle's errors / quadratic form / Schur solve (oracle/ref_lm_wrap.cpp)
# "full": the same driver over g2o's own vertices, edges, Huber kernel and base-edge templates; only the Schur complement and the
#         LDL^T under Solver::solve() are the oracle's (oracle/ref_ba_full_wrap.cpp)
# "block": as "full", plus g2o's own BlockSolver_6_3 — block allocation and Hschur pattern, buildSystem, setLambda / restoreDiagonal, the Schur
#          complement and the landmark back-substitution of solve(); only LinearSolver::solve (the sparse LDL^T) is the oracle's
#          (oracle/ref_ba_block_wrap.cpp)
@pytest.fixture(scope="module", params=["lm", "full", "block"])
def ref(oracle, request):
    live = {"lm": oracle.ref_lm, "full": oracle.ref_ba_full, "block": oracle.ref_ba_block}[request.param]
    return _Side(Recorded(oracle, __file__, live, keep={"trace"}), request.param)


def same_run(a, b):
    assert a["iters_done"] == b["iters_done"] and a["trials_total"] == b["trials_total"]
    assert len(a["trace"]) == len(b["trace"])
    for c in (0, 1, 2, 4, 5):       # iteration, lambda of the last trial, robust chi2 kept, trials, lambda handed to the next iteration
        if c == 1 and np.isnan(b["trace"][:, 1]).all():
            continue                # with the reference's own BlockSolver the last trial's lambda is not visible from outside
        assert same(a["trace"][:, c], b["trace"][:, c]), c
    assert a["chi2_initial"] == b["chi2_initial"] and a["chi2_final"] == b["chi2_final"] and a["lambda_final"] == b["lambda_final"]
    assert same(a["poses"], b["poses"]) and same(a["points"], b["points"])
    assert same(a["chi2"], b["chi2"]) and same(a["depth_pos"], b["depth_pos"])


@pytest.mark.parametrize("name,iters,robust", [("tiny", 20, True), ("small", 20, True), ("small", 10, False), ("cfg2", 15, True)])
def test_schedule_matches_reference_driver(ref, name, iters, robust):
    p = synth.make_config(name) if name != "cfg2" else synth.make_config("cfg2", P=600)
    a = ref.ba_solve(p, iterations=iters, robust=robust)
    b = ref.ref_ba_solve(p, iterations=iters, robust=robust)
    same_run(a, b)
    assert a["iters_done"] >= 3 and a["chi2_final"] < a["chi2_initial"]


def test_rejected_trials_and_nu_doubling(ref):
    """A start far from the optimum with a tiny user lambda makes the first steps overshoot: rho < 0, lambda *= nu, nu *= 2, pop."""
    p = synth.make_config("small")
    rng = np.random.default_rng(3)
    p.points = p.points + rng.normal(0, 0.6, p.points.shape)
    hit = False
    for lam in (1e-9, 1e-6, 1e-2, 1e3):
        a = ref.ba_solve(p, iterations=12, lambda_init=lam)
        b = ref.ref_ba_solve(p, iterations=12, lambda_init=lam)
        same_run(a, b)
        hit |= bool((a["trace"][:, 4] > 1).any())
    assert hit                                       # at least one run rejected a step


def test_max_trials_terminates(ref):
    """qmax == maxTrialsAfterFailure ends optimize() after that iteration (Terminate), with the state of before the iteration."""
    p = synth.make_config("small")
    rng = np.random.default_rng(4)
    p.points = p.points + rng.normal(0, 1.5, p.points.shape)
    seen = False
    for mt in (1, 2, 3):
        a = ref.ba_solve(p, iterations=10, lambda_init=1e-12, max_trials=mt)
        b = ref.ref_ba_solve(p, iterations=10, lambda_init=1e-12, max_trials=mt)
        same_run(a, b)
        seen |= a["iters_done"] < 10 and a["trace"][-1, 4] == mt
    assert seen


def test_three_strike_stop_of_the_vendored_copy(ref):
    """(iniChi - currentChi) * 1e3 < iniChi three iterations in a row ends the run (G/core/optimization_algorithm_levenberg.cpp:148-160):
    a converged problem given 30 iterations stops early, on the same iteration under both drivers."""
    p = synth.make_config("tiny")
    a = ref.ba_solve(p, iterations=30)
    b = ref.ref_ba_solve(p, iterations=30)
    same_run(a, b)
    assert a["iters_done"] < 30


def test_second_round_flags_stop_flag_and_empty(ref):
    p = synth.make_config("cfg2", P=400)
    d = np.sqrt(5.991)
    r1 = ref.ba_solve(p, iterations=5, huber_delta=d); q1 = ref.ref_ba_solve(p, iterations=5, huber_delta=d)
    same_run(r1, q1)
    out = (r1["chi2"] > 5.991) | (r1["depth_pos"] == 0)
    p2 = p.copy(); p2.poses = r1["poses"]; p2.points = r1["points"]; p2.edge_flags = (out.astype(np.uint8) | 2).astype(np.uint8)
    same_run(ref.ba_solve(p2, iterations=10, huber_delta=d, chi2_in=r1["chi2"]), ref.ref_ba_solve(p2, iterations=10, huber_delta=d, chi2_in=r1["chi2"]))
    stop = np.ones(1, np.uint8)
    same_run(ref.ba_solve(p, iterations=20, stop=stop), ref.ref_ba_solve(p, iterations=20, stop=stop))
    same_run(ref.ba_solve(p, iterations=0), ref.ref_ba_solve(p, iterations=0))
    p3 = p.copy(); p3.edge_flags = np.ones(p.E, np.uint8)          # every edge at level 1: nothing to optimise, optimize() returns -1
    a = ref.ba_solve(p3, iterations=5); b = ref.ref_ba_solve(p3, iterations=5)
    assert a["iters_done"] == b["iters_done"] == -1
