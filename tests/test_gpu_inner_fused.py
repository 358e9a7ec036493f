"""Inner iterations (Ceres' CoordinateDescentMinimizer, csrc/pxr_inner.cuh) at sizes the parity tests do not reach:
thousands of points, tracks longer than a warp, constant points and points without observations, window residency
that forces patch refetches while the points move — against the CPU oracle, or bit for bit against the same solve
where nothing has to be refetched."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from pixsfm._pixsfm import _capi, _engine
from pixsfm.util import synthetic

pytestmark = pytest.mark.gpu


def _scene(**kw):
    prob, _ = synthetic.make_ba_scene(**kw)
    ic = _capi.default_interp()
    prob.refs, _ = O.refs_compute(prob, ic)
    return prob, ic


def _drop_observations(prob, points):
    """the same problem without any observation of `points` (the patches stay, reached through obs_patch)"""
    keep = ~np.isin(prob.obs_pt, points)
    return _capi.BAProblem(prob.cam_model, prob.cam_params, prob.cam_const_mask, prob.qvec, prob.tvec, prob.img_cam,
                           prob.pose_const, prob.tvec_const_mask, prob.xyz, prob.point_const, prob.obs_img[keep],
                           prob.obs_pt[keep], prob.patches, prob.corner, prob.scale, refs=prob.refs,
                           obs_patch=np.nonzero(keep)[0].astype(np.int64))


@pytest.mark.parametrize("kind", ["many_points", "long_tracks"])
def test_inner_iterations_match_oracle_points(kind):
    if kind == "many_points":
        prob, ic = _scene(n_cams=12, n_points=3000, track_len=5, channels=32, seed=11)
    else:       # 40 observations per point: the per-point sums run over more than one warp of records
        prob, ic = _scene(n_cams=48, n_points=200, track_len=40, channels=16, seed=12)
    n = len(prob.xyz)
    prob.point_const[::7] = 1
    prob = _drop_observations(prob, np.arange(3, n, 11))
    prob.xyz += np.random.default_rng(5).normal(0, 0.004, prob.xyz.shape)
    so = _capi.default_ba_options(use_inner_iterations=1)
    h = _engine.BAHandle(prob.copy(), ic, so)
    h.debug_inner_iterations()
    h.read_params()
    p_ref = prob.copy()
    d = p_ref.desc()
    O.lib().orc_ba_inner_iterations(C.byref(d), C.byref(ic), C.byref(so))
    assert np.abs(h.problem.xyz - p_ref.xyz).max() < 1e-7
    fixed = np.zeros(n, bool)
    fixed[::7] = True
    fixed[3::11] = True
    assert np.array_equal(h.problem.xyz[fixed], prob.xyz[fixed])
    assert np.abs(p_ref.xyz[~fixed] - prob.xyz[~fixed]).max() > 1e-5    # the others did move


def test_cost_after_inner_iterations_equals_a_full_evaluation():
    """The cost after the inner iterations is summed from what the kernel left per observation; a step it made
    acceptable is then linearised by a full evaluation at the same parameters, which must give the same bits (block
    mode takes the trial cost as the new cost without re-evaluating it, so this runs the default mode)."""
    prob, ic = _scene(n_cams=10, n_points=1000, track_len=5, channels=128, seed=13, pt_sigma=0.01)
    so = _capi.default_ba_options(max_num_iterations=10, use_inner_iterations=1)
    s = _engine.ba_run(prob, ic, so)
    its = s["iterations"]
    n_inner = s["num_inner_iteration_steps"]
    assert n_inner >= 2
    x_cost, checked = its[0]["cost"], 0
    for it in its[1:n_inner + 1]:                # inner iterations run from the first iteration until they stop paying
        if it["step_is_successful"]:
            assert it["cost_change"] == x_cost - it["cost"]
            x_cost = it["cost"]
            checked += 1
    assert checked >= 1


def _run_windowed(prob, ic, so, window):
    pin = _engine.PinnedArray(prob.patches.shape, prob.patches.dtype)
    pin.array[...] = prob.patches
    q = prob.copy()
    q.patches = pin.array
    q._patches_ptr = pin.array.ctypes.data
    old = os.environ.get("PXR_RESIDENT_WINDOW")
    os.environ["PXR_RESIDENT_WINDOW"] = str(window)
    try:
        s = _engine.ba_run(q, ic, so)
    finally:
        if old is None:
            os.environ.pop("PXR_RESIDENT_WINDOW", None)
        else:
            os.environ["PXR_RESIDENT_WINDOW"] = old
    out = (s, q.xyz.copy(), q.qvec.copy(), q.tvec.copy(), q.cam_params.copy())
    pin.close()
    return out


def test_windowed_inner_iterations_refetch_and_stay_bit_identical():
    # a rough start: the inner iterations move points out of 4x4-tap windows, whose patches are then fetched whole and
    # the inner iterations run again from their starting points
    prob, ic = _scene(n_cams=10, n_points=2000, track_len=5, channels=128, seed=14, rot_sigma_deg=0.06, pt_sigma=0.012)
    so = _capi.default_ba_options(max_num_iterations=8, use_inner_iterations=1, deterministic=1)
    full = _run_windowed(prob, ic, so, 0)
    win = _run_windowed(prob, ic, so, 4)
    assert full[0]["resident_window"] == 0 and win[0]["resident_window"] == 4
    assert win[0]["resident_refetched"] > 0 and win[0]["resident_passes_repeated"] > 0
    assert win[0]["num_inner_iteration_steps"] == full[0]["num_inner_iteration_steps"] >= 1
    for a, b in zip(win[0]["iterations"], full[0]["iterations"]):
        for key in ("cost", "cost_change", "step_norm", "relative_decrease", "trust_region_radius"):
            assert a[key] == b[key], key
    assert len(win[0]["iterations"]) == len(full[0]["iterations"]) and win[0]["final_cost"] == full[0]["final_cost"]
    for u, v in zip(win[1:], full[1:]):
        assert np.array_equal(u, v)
