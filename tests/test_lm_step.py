"""GPU (-m gpu): single trust-region steps of k_lm (csrc/lm_kernel.cuh) against oracle/trf_exact_model.trf_step driven by the device's
own normal equations (mcba_linearize exports the H_ss, H_ff, W and g that k_lm reads).  The model solves (A + reg I) gn_h = g_h densely
in float64 with two refinement steps (residual in long double) and the 2-D subproblem by a bracketed secular-equation root, so what is
left between the two is the rounding of the device's Schur complement, Cholesky and substitutions: a relative error of about
cond(A + reg I) * eps.  The bar is max(1e-10, 16 cond eps).  A wrong tile, panel, frame chunk or damping term gives 1e-7 or more.

The shapes are where the reduced factorisation changes (solver.cu setup_problem, lm_kernel.cuh phase F):
  n_s = 6C [camera poses] + 6B [board poses] + (5 + nd) C [cameras] + 3BP [board points] + 12 [hand-eye]
  n_s <= 127: one CTA, the matrix in R = ceil(n_s / 16) register rotations; n_s >= 128: 32-wide blocked Cholesky over the grid
  grid: every SM when F_free * n_s >= 4096, else min(SMs, 8) CTAs;  Schur SYRK: 48 / fb frames per staged step, in frame chunks
"""
import os

import numpy as np
import pytest
from numpy.linalg import norm
from scipy.optimize._lsq.common import solve_trust_region_2d

from multical_b200 import synthetic
from multical_b200.calibration import from_scene
from multical_b200.motion import RollingFrames
from oracle.trf_exact_model import jac_scale, trf_exact, trf_step

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
CHOL_SMALL_MAX = 127              # csrc/solver_kernels.cuh
FULL_GRID_WORK = 4096             # csrc/solver.cu: F_free * n_s at or above which k_lm runs on every SM


def charuco(count, w=5, h=4):
  return ("charuco", w, h, 0.03, count)


# name: (make_scene arguments, enabled blocks, motion model, n_s, grid rule)
CASES = {
  # single CTA, one case per rotation count R = ceil(n_s / 16)
  "ns12_R1": (dict(C=2, F=4, vis=0.5, seed=101), dict(board_poses=False), None, 12, "8"),
  "ns32_R2": (dict(C=2, F=4, vis=0.5, seed=102), dict(cameras=True, board_poses=False), None, 32, "8"),           # a multiple of 16
  "ns33_R3": (dict(C=1, F=5, vis=0.6, seed=103, model="fisheye", boards=charuco(3)), dict(cameras=True), None, 33, "8"),   # one more
  "ns54_R4": (dict(C=3, F=8, vis=0.5, seed=41), dict(cameras=True), None, 54, "8"),
  "ns70_R5": (dict(C=4, F=4, vis=0.3, seed=105), dict(cameras=True), None, 70, "8"),
  "ns86_R6": (dict(C=5, F=4, vis=0.3, seed=106), dict(cameras=True), None, 86, "8"),
  "ns102_R7": (dict(C=6, F=4, vis=0.3, seed=107), dict(cameras=True), None, 102, "8"),
  "ns127_R8": (dict(C=5, F=4, vis=0.5, seed=108, model="thin_prism", boards=charuco(2)), dict(cameras=True), None, 127, "8"),
  # blocked, 32-wide panels
  "ns128": (dict(C=8, F=3, vis=0.3, seed=109), dict(cameras=True, board_poses=False), None, 128, "8"),            # panels exact
  "ns129_full": (dict(C=7, F=35, vis=0.4, seed=110, model="fisheye", boards=charuco(4)), dict(cameras=True), None, 129, "full"),
  "ns150": (dict(C=9, F=4, vis=0.12, seed=11, rig="dome"), dict(cameras=True), None, 150, "8"),
  "ns160_fixed_motion": (dict(C=10, F=4, vis=0.3, seed=111), dict(cameras=True, board_poses=False, motion=False), None, 160, "8"),
  "ns161_rolling": (dict(C=5, F=7, vis=0.5, seed=112, model="tilted", boards=charuco(6)), dict(cameras=True), "rolling", 161, "8"),
  "ns286_full": (dict(C=16, F=15, vis=0.3, seed=113, rig="dome", boards=("cube", 10, 10, 0.040, 5)), dict(cameras=True), None, 286, "full"),
  "ns1030_full": (dict(C=64, F=4, vis=0.10, seed=5, rig="dome"), dict(cameras=True), None, 1030, "full"),
}


def make(name, scene=None):
  """(engine with the case uploaded, state at x0) + a description of the launch shape k_lm gets for it."""
  kw, enabled, motion, n_s, grid = CASES[name] if name in CASES else (None, dict(cameras=True), None, None, None)
  scene = synthetic.make_scene(**kw) if scene is None else scene
  calib = from_scene(scene)
  if motion == "rolling":
    rng = np.random.default_rng(7)
    start = scene["init"]["frame_poses"]
    end = synthetic.to_matrix(synthetic.from_matrix(start) + 1e-3 * rng.standard_normal((scene["F"], 6)))
    calib = calib.copy(motion=RollingFrames(start, end, scene["frame_valid"], [str(i) for i in range(scene["F"])]))
  calib = calib.enable(**enabled)
  eng = calib._upload(calib.inliers)
  fb = 12 if motion == "rolling" else 6
  F_free = scene["F"] if calib.optimize["motion"] else 0
  shape = dict(n_s=eng.num_params - fb * F_free, F_free=F_free, fb=fb)
  shape["path"] = "single" if shape["n_s"] <= CHOL_SMALL_MAX else "blocked"
  shape["grid"] = "full" if max(F_free, 1) * shape["n_s"] >= FULL_GRID_WORK else "8"
  if n_s is not None:
    assert (shape["n_s"], shape["grid"]) == (n_s, grid), (name, shape)
  return eng, shape


def cost_at(eng, x):
  return eng.residuals(x, with_cost=True)[1]


def step_error(dx, scale_inv, model):
  """relative error of the device's scaled step against the model's, and the bar it has to meet."""
  err = norm(dx * scale_inv - model["step_h"]) / norm(model["step_h"])
  return err, max(1e-10, 16 * model["cond"] * EPS)


def check_2d_against_scipy(model, Delta):
  """The model's secular-equation solve of the 2-D subproblem against scipy's solve_trust_region_2d.  Interior: both are the Newton
  point of a 2 x 2 positive definite system (Cholesky there, eigenvalues here), equal to ~cond(B_S) eps.  Boundary: scipy takes the
  best real root of a quartic from np.roots (companion-matrix eigenvalues), whose accuracy falls with the spread of the quartic's
  coefficients (Delta^2 against the entries of B_S); 1e-6 is a bound it meets with room on these problems, not a statement about
  either solve's precision -- that is the job of the 1e-10 comparison with the device."""
  p_ref, _ = solve_trust_region_2d(model["B_S"], model["g_S"], Delta)
  tol = 1e-6 if model["boundary"] else 1e-10
  assert norm(p_ref - model["p_S"]) <= tol * norm(model["p_S"]), (p_ref, model["p_S"], model["boundary"])


def first_step(eng, x0):
  """The model's first step at x0 and the device's solve with max_nfev=2 (one trial)."""
  JtJ, g, _ = eng.linearize(x0)                       # leaves the device state at x0
  scale_inv = jac_scale(JtJ)
  Delta = norm(x0 * scale_inv) or 1.0
  model = trf_step(JtJ, g, x0, Delta, scale_inv)
  res = eng.solve(max_nfev=2)
  return model, scale_inv, Delta, res, eng.param_vec - x0


def check_first_step(name):
  eng, shape = make(name)
  x0 = eng.param_vec
  cost0 = cost_at(eng, x0)
  model, scale_inv, Delta, res, dx = first_step(eng, x0)
  check_2d_against_scipy(model, Delta)
  assert res.chol_retries == 0
  assert [row[:2] for row in res.log[:2]] == [(0, 1), (1, 2)], res.log       # the trial was taken
  err, tol = step_error(dx, scale_inv, model)
  assert err <= tol, f"{name} {shape}: step_h relative error {err:.3e} > {tol:.3e} (cond {model['cond']:.3e}, reg {model['reg']:.3e})"
  _, _, _, red, sn, _ = res.log[1]
  assert abs(sn - norm(model["step"])) <= tol * norm(model["step"]), (sn, norm(model["step"]))
  red_model = cost0 - cost_at(eng, x0 + model["step"])
  assert red_model > 0
  assert abs(red - red_model) <= 1e-9 * red_model + 1e-14 * cost0, (red, red_model, cost0)
  return err, tol, model


@pytest.mark.parametrize("name", list(CASES))
def test_first_step_matches_the_refined_dense_model(name):
  """Linearise at x0, one trial step (max_nfev=2): the step, its norm in the log and the cost reduction against the model."""
  check_first_step(name)


def rejected_then_boundary(name, n_poses, seed, scale):
  """A start far from the optimum: the first `n_poses` parameters (camera, board and frame twists, canonical order) moved by `scale`
  (radians, metres) times a standard normal.  Rejections are decided from the model's own costs: the first trial at Delta0 must raise
  the cost; the retries shrink Delta to 0.25 ||step_h|| (update_tr_radius) until a trial is accepted.  Returns everything the device
  must reproduce."""
  eng, shape = make(name)
  x0 = eng.param_vec
  x0[:n_poses] += scale * np.random.default_rng(seed).standard_normal(n_poses)
  JtJ, g, _ = eng.linearize(x0)
  cost0 = cost_at(eng, x0)
  scale_inv = jac_scale(JtJ)
  Delta0 = Delta = norm(x0 * scale_inv) or 1.0
  nfev, trials = 1, []
  while True:
    model = trf_step(JtJ, g, x0, Delta, scale_inv, reg_Delta=Delta0)
    nfev += 1
    red = cost0 - cost_at(eng, x0 + model["step"])
    trials.append((Delta, model, red))
    if red > 0 or nfev > 6: break
    Delta = 0.25 * norm(model["step_h"])
  return eng, shape, x0, cost0, scale_inv, nfev, trials


def test_rejected_trial_then_boundary_step_on_the_blocked_path():
  """A start perturbed so far (fixed seed) that the first trial raises the cost: the device must reject it, shrink the radius to
  0.25 ||step_h|| and take the retried step, which lies on the boundary.  The log shows the retry (nfev moves, the iteration does not);
  the accepted step is compared with the model at the first-step tolerance."""
  # ns150: 9 cameras, one board, 4 frames -> 6 * (9 + 1 + 4) pose parameters ahead of the 9 x 10 intrinsics
  eng, shape, x0, cost0, scale_inv, nfev, trials = rejected_then_boundary("ns150", n_poses=84, seed=4, scale=0.3)
  assert shape["path"] == "blocked"
  assert len(trials) >= 2 and trials[0][2] < 0 and trials[-1][2] > 0, [t[2] for t in trials]
  Delta, model, red_model = trials[-1]
  assert model["boundary"] and abs(norm(model["step_h"]) - Delta) <= 1e-12 * Delta
  check_2d_against_scipy(model, Delta)
  eng.set_param_vec(x0)
  res = eng.solve(max_nfev=nfev)
  assert res.chol_retries == 0
  assert [row[:2] for row in res.log[:2]] == [(0, 1), (1, nfev)], res.log      # nfev moved by len(trials), the iteration by one
  err, tol = step_error(eng.param_vec - x0, scale_inv, model)
  assert err <= tol, f"boundary step_h relative error {err:.3e} > {tol:.3e} (cond {model['cond']:.3e}, Delta {Delta:.3e})"
  _, _, _, red, sn, _ = res.log[1]
  assert abs(sn - norm(model["step"])) <= tol * norm(model["step"])
  assert abs(red - red_model) <= 1e-9 * red_model + 1e-14 * cost0, (red, red_model)


def near(a, b, rel=1e-6):
  return abs(a - b) <= rel * abs(b)


def comparable_prefix(trace, ftol, xtol):
  """Number of trial steps of the model whose control decisions are not within 1e-6 relative of a threshold: the ratio against 0.25
  and 0.75, ||step_h|| against 0.95 Delta, the ftol and xtol tests, and the sign of the reduction (against the rounding of two costs)."""
  for k, t in enumerate(trace):
    if (near(t["ratio"], 0.25) or near(t["ratio"], 0.75) or near(t["step_h_norm"], 0.95 * t["Delta"])
        or near(t["reduction"], ftol * t["cost"]) or near(t["step_norm"], xtol * (xtol + t["x_norm"]))
        or abs(t["reduction"]) <= 1e-12 * t["cost"]):
      return k
  return len(trace)


@pytest.mark.parametrize("name", ["ns150", "ns286_full", "ns161_rolling"])
def test_iteration_table_matches_the_model_on_device_normal_equations(name):
  """The whole solve: the model (trf_exact with lin = the device's normal equations at the model's own iterates, cost of a trial from
  the device's residuals) against eng.solve, row by row, up to the first control decision within 1e-6 of its threshold.

  Each row is held to 1e-10 (cost) and 1e-8 (reduction, step norm, optimality) of its own value, plus an absolute part on the scale of
  the first rows.  The two solves walk their own iterates, which after the first step differ by that step's rounding (1e-12 .. 1e-11 of
  it on these scenes); the first step takes the cost down by three to four orders of magnitude, so what a later row inherits from it is
  a fixed amount on the scale of the initial cost, step and gradient, not a fraction of the row's own (much smaller) values."""
  ftol = xtol = gtol = 1e-10
  eng, shape = make(name)
  x0 = eng.param_vec
  trace = []
  _, _, _, _, _, rows = trf_exact(lambda x: eng.residuals(x), None, x0, ftol=ftol, xtol=xtol, gtol=gtol, max_nfev=14,
                                  lin=lambda x: eng.linearize(x), trace=trace)
  eng.set_param_vec(x0)
  res = eng.solve(ftol=ftol, xtol=xtol, gtol=gtol, max_nfev=14)
  assert res.chol_retries == 0
  n_trials = comparable_prefix(trace, ftol, xtol)
  # a row is comparable when every trial before it was: row k's nfev counts the trials that led to it
  n_rows = sum(1 for r in rows if r[1] - 1 <= n_trials)
  assert n_rows >= 5, (n_rows, n_trials, len(rows))
  assert len(res.log) >= n_rows
  c0, sn1, g0 = rows[0][2], rows[1][4], rows[0][5]
  for (it, nf, c, red, sn, gn), (it2, nf2, c2, red2, sn2, gn2) in zip(res.log[:n_rows], rows[:n_rows]):
    assert (it, nf) == (it2, nf2), (res.log[:n_rows], rows[:n_rows])
    assert abs(c - c2) <= 1e-10 * c2 + 1e-12 * c0, (it, c, c2)
    if red2 is not None:
      assert abs(red - red2) <= 1e-8 * abs(red2) + 2e-12 * c0, (it, red, red2)
      assert abs(sn - sn2) <= 1e-8 * sn2 + 1e-8 * sn1, (it, sn, sn2)
    assert abs(gn - gn2) <= 1e-8 * gn2 + 1e-8 * g0, (it, gn, gn2)


def test_configs4_first_step_at_full_size():
  """BASELINE configs[4] (synthetic cfg4: 16 cameras x 1000 frames, five cube boards, n_s = 286, n = 6286) at the launch shape bench.py
  times: every SM, frame chunks of the full machine.  The dense model is seconds of numpy at this size."""
  scene = synthetic.make_workload("cfg4")
  eng, shape = make("cfg4", scene=scene)
  assert (shape["n_s"], shape["F_free"], shape["grid"]) == (286, 1000, "full")
  x0 = eng.param_vec
  cost0 = cost_at(eng, x0)
  model, scale_inv, Delta, res, dx = first_step(eng, x0)
  assert res.chol_retries == 0 and [row[:2] for row in res.log[:2]] == [(0, 1), (1, 2)]
  err, tol = step_error(dx, scale_inv, model)
  assert err <= tol, f"cfg4: step_h relative error {err:.3e} > {tol:.3e} (cond {model['cond']:.3e})"
  red_model = cost0 - cost_at(eng, x0 + model["step"])
  assert abs(res.log[1][3] - red_model) <= 1e-9 * red_model + 1e-14 * cost0
