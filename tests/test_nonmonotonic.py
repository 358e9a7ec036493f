"""use_nonmonotonic_steps (ceres::Solver::Options; the reference's configs/default.yaml switches it on for KA, BA and
QKA): the oracle's restatement of ceres' TrustRegionStepEvaluator, the reference YAML files (configs/default.yaml and
low_memory.yaml, kept under tests/golden/configs/) taken as far as the solver options of every optimizer, and (GPU) the
device LM drivers against the oracle with the option on."""
import os

import numpy as np
import pytest

import oracle_lib as O
from pixsfm._pixsfm import _capi
from pixsfm.util import synthetic

REF_CONFIGS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "configs")


def _hard_ba_problem(seed=4):
    """a start far enough from the optimum that LM takes both accepted and rejected steps"""
    prob, _ = synthetic.make_ba_scene(n_cams=5, n_points=40, track_len=4, channels=16, seed=seed, pt_sigma=0.06,
                                      rot_sigma_deg=0.3, t_sigma=0.02)
    ic = _capi.default_interp()
    prob.refs, _ = O.refs_compute(prob, ic)
    return prob, ic


def test_monotonic_evaluator_is_the_old_rule_and_nonmonotonic_returns_the_best_iterate():
    prob, ic = _hard_ba_problem()
    base = dict(max_num_iterations=25, use_inner_iterations=0)
    p_m, p_n = prob.copy(), prob.copy()
    s_m = O.ba_solve(p_m, ic, _capi.default_ba_options(**base))
    s_n = O.ba_solve(p_n, ic, _capi.default_ba_options(use_nonmonotonic_steps=1, max_consecutive_nonmonotonic_steps=10, **base))
    # the option is exercised: some accepted steps of the non-monotonic run INCREASE the cost
    assert any(i["step_is_successful"] and i["cost_change"] < 0 for i in s_n["iterations"])
    for s in (s_m, s_n):
        assert s["final_cost"] <= s["initial_cost"]
        assert s["final_cost"] == min(i["cost"] for i in s["iterations"] if i["step_is_successful"] or i["iteration"] == 0)
    # monotonic: every accepted step lowers the cost
    costs = [i["cost"] for i in s_m["iterations"] if i["step_is_successful"]]
    assert all(b < a for a, b in zip([s_m["initial_cost"]] + costs, costs))
    # the parameters handed back are the lowest-cost iterate (ceres writes x back only when it improves on the minimum)
    so = _capi.default_ba_options(**base)
    assert abs(O.ba_evaluate(p_n, ic, so)["cost"] - s_n["final_cost"]) <= 1e-12 * s_n["final_cost"]
    assert abs(O.ba_evaluate(p_m, ic, so)["cost"] - s_m["final_cost"]) <= 1e-12 * s_m["final_cost"]


@pytest.mark.parametrize("name", ["default.yaml", "low_memory.yaml"])
def test_reference_yaml_reaches_the_solver_options(name):
    """ADVICE r1: PixSfM(<reference yaml>) must not only construct but also yield solver options for every optimizer"""
    import yaml
    from pixsfm._pixsfm._bundle_adjustment import solver_options_from
    from pixsfm.localization.main import QueryBundleAdjuster, QueryKeypointAdjuster
    from pixsfm.refine_colmap import PixSfM
    path = os.path.join(REF_CONFIGS, name)
    sfm = PixSfM(path)
    raw = yaml.safe_load(open(path))
    for part, base in ((sfm.conf.KA, _capi.default_ka_options()), (sfm.conf.BA, _capi.default_ba_options())):
        opt = part.optimizer
        so = solver_options_from(dict(opt.loss), dict(opt.solver), base)
        assert so.max_num_iterations == opt.solver.max_num_iterations
        assert so.use_nonmonotonic_steps == int(bool(opt.solver.use_nonmonotonic_steps))
        if so.use_nonmonotonic_steps:
            assert so.max_consecutive_nonmonotonic_steps == opt.solver.max_consecutive_nonmonotonic_steps
    if name == "default.yaml":
        assert raw["mapping"]["BA"]["optimizer"]["solver"]["use_nonmonotonic_steps"] is True
        so = solver_options_from(dict(sfm.conf.BA.optimizer.loss), dict(sfm.conf.BA.optimizer.solver), _capi.default_ba_options())
        assert so.use_nonmonotonic_steps == 1 and so.max_consecutive_nonmonotonic_steps == 10 and so.use_inner_iterations == 1
        from pixsfm.refine_colmap import _resolve_references
        loc_conf = _resolve_references(raw["localization"], raw)
        qka = QueryKeypointAdjuster(loc_conf["QKA"])
        qba = QueryBundleAdjuster(loc_conf["QBA"])
        assert qka.solver.solver_options().use_nonmonotonic_steps == 1
        assert qba.solver.solver_options().use_nonmonotonic_steps == 0


@pytest.mark.gpu
@pytest.mark.parametrize("inner", [0, 1])
def test_gpu_ba_with_nonmonotonic_steps_matches_the_oracle(inner):
    """Non-monotonic trajectories on a far-off start are chaotic: the ORACLE's own costs move by up to 1e-5 relative when
    its input is perturbed by 1e-13 (measured below, per iteration).  The GPU has to stay within 10x that envelope (and
    1e-6 where the envelope is tighter), with the same accept / reject sequence."""
    from pixsfm._pixsfm import _engine
    prob, _ = synthetic.make_ba_scene(n_cams=5, n_points=40, track_len=4, channels=16, seed=5, pt_sigma=0.03,
                                      rot_sigma_deg=0.15, t_sigma=0.01)
    ic = _capi.default_interp()
    prob.refs, _ = O.refs_compute(prob, ic)
    so = _capi.default_ba_options(max_num_iterations=14, use_inner_iterations=inner, use_nonmonotonic_steps=1,
                                  max_consecutive_nonmonotonic_steps=10)
    p_cpu, p_eps, p_gpu = prob.copy(), prob.copy(), prob.copy()
    p_eps.xyz = p_eps.xyz + 1e-13
    s_cpu = O.ba_solve(p_cpu, ic, so)
    s_eps = O.ba_solve(p_eps, ic, so)
    assert any(i["step_is_successful"] and i["cost_change"] < 0 for i in s_cpu["iterations"])      # the option is exercised
    env = [max(1e-6, 10 * abs(a["cost"] - b["cost"]) / abs(a["cost"])) for a, b in zip(s_cpu["iterations"], s_eps["iterations"])]
    env = np.maximum.accumulate(env)
    s_gpu = _engine.ba_run(p_gpu, ic, so)
    assert len(s_gpu["iterations"]) == len(s_cpu["iterations"])
    for ig, ir, tol in zip(s_gpu["iterations"], s_cpu["iterations"], env):
        assert ig["step_is_successful"] == ir["step_is_successful"]
        assert abs(ig["cost"] - ir["cost"]) <= tol * abs(ir["cost"])
    assert abs(s_gpu["final_cost"] - s_cpu["final_cost"]) <= env[-1] * s_cpu["final_cost"]
    ptol = max(1e-6, 10 * np.abs(p_eps.xyz - p_cpu.xyz).max())
    assert np.abs(p_gpu.xyz - p_cpu.xyz).max() < ptol and np.abs(p_gpu.qvec - p_cpu.qvec).max() < ptol
    # what comes back is the best iterate
    assert abs(_engine.BAHandle(p_gpu, ic, so).evaluate()["cost"] - s_gpu["final_cost"]) <= 1e-9 * s_gpu["final_cost"]


@pytest.mark.gpu
def test_gpu_ka_with_nonmonotonic_steps_matches_the_oracle():
    from ka_util import make_ka_problem
    from pixsfm._pixsfm import _engine
    prob, sc, lab = make_ka_problem(n_images=6, n_tracks=40, track_len=4, channels=128, seed=2, kp_sigma=2.0, bound=4.0,
                                    max_per_problem=20)
    ic = _capi.default_interp()
    so = _capi.default_ka_options(use_nonmonotonic_steps=1, max_consecutive_nonmonotonic_steps=10)
    p_cpu, p_gpu = prob.copy(), prob.copy()
    c0, c1 = O.ka_solve(p_cpu, ic, so)
    s = _engine.ka_run(p_gpu, ic, so)
    assert abs(s["initial_cost"] - c0) <= 1e-9 * c0 and abs(s["final_cost"] - c1) <= 1e-6 * c1 and c1 < c0
    assert np.abs(p_gpu.keypoints - p_cpu.keypoints).max() < 1e-5
