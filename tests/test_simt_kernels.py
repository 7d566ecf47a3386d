"""CPU (-m "not gpu"): the REAL CUDA kernels and the REAL host driver of multical_b200/csrc, executed by the SIMT interpreter of
tests/simt (every CUDA thread a fiber, blocks one after the other) behind the same C-ABI, against the same oracle / golden
assertions as the GPU suite.  The test functions are the ones of tests/test_gpu_parity.py and tests/test_gpu_table.py -- imported,
not copied -- with the ctypes binding pointed at tests/simt/build/libmcba_simt.so for the duration of each test.

What this proves without a GPU: indexing, math, shared-memory layouts, warp-collective usage (full-mask discipline, barrier
placement -- a divergent barrier aborts the interpreter) and the host-side plumbing of every kernel launched by these tests.
What it cannot prove: anything about concurrency (blocks and fibers run deterministically) or speed; that is the GPU suite's job.
The library is test infrastructure: the product (multical_b200/_native.py) never loads it.
"""

import os
import pytest

import test_gpu_parity as gp
import test_gpu_table as gt
import test_gpu_motion as gm
import test_gpu_pnp as gn
import test_lm_step as ls
from multical_b200 import _native, calibration


@pytest.fixture(scope="session")
def simt_library():
  import simt                     # tests/simt/__init__.py (tests/ is on sys.path: pytest rootdir/conftest import mode)
  return simt.build()


@pytest.fixture(autouse=True)
def on_the_interpreter(simt_library, monkeypatch):
  """Point the ctypes binding at the interpreter build for one test; engines are per-library, so the cache is swapped as well."""
  monkeypatch.setattr(_native, "LIB_PATH", simt_library)
  monkeypatch.setattr(_native, "_lib", None)
  monkeypatch.setattr(_native, "_allow_interpreter", True)
  monkeypatch.setattr(calibration, "_engines", {})
  monkeypatch.delenv("SIMT_SMS", raising=False)
  yield
  for eng in calibration._engines.values(): eng.close()


# ---- tests/test_gpu_parity.py on the interpreter (the two large-scene property tests stay GPU-only: minutes of fiber switching)
test_residuals_match_reference_golden_and_oracle = gp.test_residuals_match_reference_golden_and_oracle
test_reprojection_error_over_valid = gp.test_reprojection_error_over_valid
test_normal_equations_match_finite_differences = gp.test_normal_equations_match_finite_differences
test_converged_solution_matches_dense_exact_oracle = gp.test_converged_solution_matches_dense_exact_oracle


@pytest.mark.parametrize("loss", ["soft_l1", "huber", "cauchy"])          # arctan (slow to converge: 45 s of fiber switching) stays GPU-only
def test_robust_losses_follow_scipy(loss):
  gp.test_robust_losses_follow_scipy(loss)


test_outlier_loop_matches_reference_semantics = gp.test_outlier_loop_matches_reference_semantics
test_fixed_blocks_and_fix_aspect = gp.test_fixed_blocks_and_fix_aspect
test_bad_inputs_raise_like_the_reference = gp.test_bad_inputs_raise_like_the_reference
test_device_packing_equals_host_packing = gp.test_device_packing_equals_host_packing
test_empty_and_ragged_inputs = gp.test_empty_and_ragged_inputs
test_board_points_as_parameters = gp.test_board_points_as_parameters
test_iteration_table_matches_the_trf_model = gp.test_iteration_table_matches_the_trf_model
test_degenerate_block_selections = gp.test_degenerate_block_selections
test_many_cameras_use_the_cooperative_blocked_reduced_solve = gp.test_many_cameras_use_the_cooperative_blocked_reduced_solve
test_frame_count_that_ends_a_syrk_chunk_in_a_partial_step = gp.test_frame_count_that_ends_a_syrk_chunk_in_a_partial_step
if os.environ.get("MCBA_SIMT_FULL") == "1":      # three minutes on the interpreter (n_s = 1030): opt-in, the GPU suite always runs it
  test_sixty_four_cameras_configs4_shape = gp.test_sixty_four_cameras_configs4_shape
test_two_identical_solves_agree_bit_for_bit = gp.test_two_identical_solves_agree_bit_for_bit

def test_more_views_per_frame_and_more_boards_than_the_staged_tables_hold():
  """k_linearize stages a frame's view records (up to 96) and the board pose tables (up to 8) in shared memory and reads them from
  global memory beyond that (csrc/linearize.cuh LIN_MAXV, LIN_MAXB).  12 cameras x 9 boards: 108 views per frame, 9 board tables --
  both fall-backs at once.  Residuals against the oracle, normal equations against finite differences of the oracle."""
  import numpy as np
  from scipy.optimize._numdiff import approx_derivative, group_columns
  from multical_b200 import synthetic
  from multical_b200.calibration import from_scene
  from oracle.ba_oracle import Problem
  scene = synthetic.make_scene(C=12, F=2, vis=0.9, seed=3, boards=("charuco", 5, 4, 0.03, 9))
  assert (scene["valid"].any(axis=-1).sum(axis=(0, 2)) > 96).all() and scene["B"] == 9
  calib = from_scene(scene).enable(cameras=True)
  prob = Problem.from_scene(scene, optimize=dict(cameras=True))
  eng = calib._upload(calib.inliers)
  x = prob.param_vec
  assert np.abs(eng.residuals(x) - prob.residuals(x)).max() < 1e-9
  S = prob.sparsity_matrix()
  J = approx_derivative(prob.residuals, x, method="3-point", sparsity=(S, group_columns(S))).toarray()
  r = prob.residuals(x)
  H, g = J.T @ J, J.T @ r
  JtJ, Jtr, cost = eng.linearize(x)
  nrm = np.sqrt(np.outer(np.diag(H), np.diag(H)))
  live = nrm > 0
  assert (np.abs(JtJ - H)[live] / nrm[live]).max() < 1e-6
  assert np.abs(Jtr - g).max() < 1e-6 * np.abs(g).max()
  assert abs(cost - 0.5 * r @ r) < 1e-12 * cost


def test_rolling_frames_with_a_frame_count_that_ends_in_a_partial_syrk_step():
  """Rolling frames eliminate a 12 x 12 block per frame and the Schur SYRK stages 4 of them per step: 19 frames = 5 steps, the last one
  partial, in a stage that held an earlier step (the frame-count pattern of test_frame_count_that_ends_a_syrk_chunk_in_a_partial_step for
  FB = 12).  Residuals against the oracle, converged cost against scipy's dense exact trust region on the oracle's residuals."""
  import numpy as np
  from scipy import optimize
  from scipy.optimize._numdiff import approx_derivative, group_columns
  from multical_b200 import synthetic
  from multical_b200.calibration import from_scene
  from multical_b200.motion import RollingFrames
  from oracle.ba_oracle import Problem
  scene = synthetic.make_scene(C=2, F=19, vis=0.3, seed=5)
  rng = np.random.default_rng(7)
  start = scene["init"]["frame_poses"]
  end = synthetic.to_matrix(synthetic.from_matrix(start) + 1e-3 * rng.standard_normal((scene["F"], 6)))
  enabled = dict(cameras=True, camera_poses=True, board_poses=True, motion=True)
  prob = Problem.from_scene(scene, optimize=enabled, motion="rolling", frame_poses_end=end, image_size=scene["image_size"])
  calib = from_scene(scene).copy(motion=RollingFrames(start, end, scene["frame_valid"], [str(i) for i in range(scene["F"])])).enable(**enabled)
  eng = calib._upload(calib.inliers)
  assert eng.num_params == prob.param_vec.size
  assert np.abs(eng.residuals(prob.param_vec) - prob.residuals(prob.param_vec)).max() < 1e-9
  S = prob.sparsity_matrix(); groups = group_columns(S)
  jac = lambda x: approx_derivative(prob.residuals, x, method="3-point", sparsity=(S, groups)).toarray()
  ref = optimize.least_squares(prob.residuals, prob.param_vec, jac=jac, x_scale="jac", ftol=1e-13, xtol=1e-13, gtol=1e-13,
                               max_nfev=200, method="trf", tr_solver="exact")
  out = calib.bundle_adjust(tolerance=1e-13, xtol=1e-13, gtol=1e-13, max_iterations=200)
  assert abs(out.last_solve.cost - ref.cost) <= 1e-8 * ref.cost, (out.last_solve.cost, ref.cost)


# ---- tests/test_gpu_table.py on the interpreter
test_table_errors_ranks_and_reject_are_numpy_on_the_same_errors = gt.test_table_errors_ranks_and_reject_are_numpy_on_the_same_errors
test_resident_adjust_outliers_equals_host_loop = gt.test_resident_adjust_outliers_equals_host_loop
test_table_from_detections_is_make_point_table = gt.test_table_from_detections_is_make_point_table
test_table_state_machine_refuses_stale_errors = gt.test_table_state_machine_refuses_stale_errors
test_outlier_steps_match_reference_golden = gt.test_outlier_steps_match_reference_golden
test_workspace_calibrate_is_enable_plus_the_outlier_loop = gt.test_workspace_calibrate_is_enable_plus_the_outlier_loop

# ---- tests/test_gpu_motion.py on the interpreter (RollingFrames, HandEye)
test_motion_layout_residuals_and_errors_match_reference_golden = gm.test_layout_residuals_and_errors_match_reference_golden
test_motion_normal_equations_match_finite_differences = gm.test_normal_equations_match_finite_differences
test_motion_converged_solution_matches_dense_exact_oracle = gm.test_converged_solution_matches_dense_exact_oracle
test_motion_iteration_table_matches_the_trf_model = gm.test_iteration_table_matches_the_trf_model
test_rolling_projection_without_measurements_iterates_like_the_reference = gm.test_rolling_projection_without_measurements_iterates_like_the_reference
test_motion_state_entry_points_refuse_the_wrong_problem = gm.test_motion_state_entry_points_refuse_the_wrong_problem
test_motion_mirror_classes_keep_the_reference_semantics = gm.test_mirror_classes_keep_the_reference_semantics
test_hand_eye_calibration_wrapper_from_arm_poses = gm.test_hand_eye_calibration_wrapper_from_arm_poses
test_motion_board_points_as_parameters_under_a_motion_model = gm.test_board_points_as_parameters_under_a_motion_model
test_motion_outlier_loop_on_the_resident_table_equals_the_host_loop = gm.test_outlier_loop_on_the_resident_table_equals_the_host_loop

# ---- tests/test_gpu_pnp.py on the interpreter (batched board-pose initialisation)
test_pnp_pose_table_matches_reference_golden = gn.test_pose_table_matches_reference_golden
test_pnp_every_camera_model_against_opencv = gn.test_every_camera_model_against_opencv
test_pnp_minimum_detections_rule_and_bad_inputs = gn.test_minimum_detections_rule_and_bad_inputs
test_pnp_april_grid_style_ids_use_the_tag_grid = gn.test_april_grid_style_ids_use_the_tag_grid


# ---- tests/test_lm_step.py on the interpreter (one k_lm step against the refined dense model; n_s = 129 and 161 at three grid sizes below)
_GRID_CASES = ("ns129_full", "ns161_rolling")


@pytest.mark.parametrize("name", [c for c in ls.CASES if c not in _GRID_CASES and (c != "ns1030_full" or os.environ.get("MCBA_SIMT_FULL") == "1")])
def test_lm_first_step_matches_the_refined_dense_model(name):
  ls.check_first_step(name)


@pytest.mark.parametrize("sms", [1, 3, None])
@pytest.mark.parametrize("name", _GRID_CASES)
def test_lm_first_step_at_three_grid_sizes(name, sms, monkeypatch):
  """SIMT_SMS (the SM count the interpreter reports, read when the context is created): 1 -> k_lm on one CTA, where one CTA also works
  off every trailing-update tile of the blocked factorisation; 3 -> CTA 0 plus two helpers; default (148, a B200) -> the launch shape of
  the GPU suite."""
  if sms is not None: monkeypatch.setenv("SIMT_SMS", str(sms))
  ls.check_first_step(name)


test_lm_rejected_trial_then_boundary_step_on_the_blocked_path = ls.test_rejected_trial_then_boundary_step_on_the_blocked_path
test_lm_iteration_table_matches_the_model_on_device_normal_equations = ls.test_iteration_table_matches_the_model_on_device_normal_equations


def test_the_product_refuses_the_interpreter_build(simt_library, monkeypatch):
  """Pointing the product at the interpreter library (e.g. through MCBA_LIB) must fail loudly: there is no CPU path."""
  monkeypatch.setattr(_native, "_allow_interpreter", False)
  monkeypatch.setattr(_native, "_lib", None)
  with pytest.raises(_native.NativeError, match="no CPU path"):
    _native.load()


def test_every_kernel_launch_and_shared_declaration_is_translated(simt_library):
  """The interpreter build is a textual translation of csrc/: no `<<<`, `__shared__` or inline PTX may survive it, and every launch of
  the sources must have become exactly one simt::launch."""
  import os, re
  import simt
  n_src = n_out = 0
  for f in simt.sources():
    src = open(os.path.join(simt.CSRC, f)).read()
    out = open(os.path.join(simt.OUT, f[:-3] + ".cpp" if f.endswith(".cu") else f)).read()
    n_src += src.count("<<<"); n_out += out.count("simt::launch(")
    assert "<<<" not in out and "asm volatile" not in out and not re.search(r"\b__shared__\b", out), f
  assert n_src == n_out and n_src > 30


# ---- the duck-typing claim: multical_b200.calibration.Calibration over the REFERENCE's own objects (build container only) ------------
def _reference():
  import os, sys
  sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "refshim"))
  import loader
  return loader if loader.available() else None


@pytest.mark.skipif(_reference() is None, reason="reference tree only exists in the build container")
@pytest.mark.parametrize("motion", ["static", "rolling", "hand_eye"])
def test_calibration_over_the_reference_objects(motion):
  """INTEGRATION.md A: swapping the class is enough -- the reference's ParamList / Camera / PoseSet / Table / motion-model objects go into
  this package's Calibration unchanged; projections equal the reference's own, and bundle_adjust returns reference objects again."""
  import numpy as np
  from multical_b200 import synthetic
  from multical_b200.calibration import Calibration
  loader = _reference()
  ref = loader.load()
  scene = synthetic.make_scene(C=2, F=5, vis=0.4, seed=77)
  spec = None
  if motion == "rolling":
    end = scene["init"]["frame_poses"].copy(); end[:, :3, 3] += 0.005
    spec = ("rolling", end)
  elif motion == "hand_eye":
    spec = ("hand_eye", scene["init"]["frame_poses"], np.eye(4), np.eye(4))          # arm poses = frame estimates, identity hand-eye pair
  rc = loader.build_calibration(ref, scene, motion=spec)
  if motion == "hand_eye": rc = rc.enable(camera_poses=False, cameras=False)
  else: rc = rc.enable(cameras=True)
  mine = Calibration(rc.cameras, rc.boards, rc.point_table, rc.camera_poses, rc.board_poses, rc.motion, optimize=rc.optimize)
  assert np.abs(np.asarray(mine.param_vec) - np.asarray(rc.param_vec)).max() < 1e-12
  ok = np.asarray(rc.reprojected.valid) & np.asarray(rc.point_table.valid)
  assert np.abs(np.asarray(mine.reprojected.points)[ok] - np.asarray(rc.reprojected.points)[ok]).max() < 1e-9
  assert np.abs(np.asarray(mine.reprojection_error) - np.asarray(rc.reprojection_error)).max() < 1e-9
  out = mine.bundle_adjust(max_iterations=10)
  assert type(out.motion) is type(rc.motion) and type(out.cameras[0]) is type(rc.cameras[0])
  r = (np.asarray(out.reprojected.points) - np.asarray(out.point_table.points))[np.asarray(out.inliers)]
  assert abs(0.5 * float(np.sum(r ** 2)) - out.last_solve.cost) <= 1e-9 * out.last_solve.cost
  assert out.last_solve.cost < 0.5 * float(np.sum(((np.asarray(rc.reprojected.points) - np.asarray(rc.point_table.points))[np.asarray(rc.inliers)]) ** 2))


@pytest.mark.parametrize("motion", ["static", "rolling", "hand_eye"])
def test_calibration_matches_the_reference_calibration_golden(motion):
  """The comparisons of test_calibration_over_the_reference_objects against what the reference's own Calibration computed on the same
  scene (tests/golden/make_golden.py reference_calibration_cases), with this package's mirror objects in place of the reference's:
  parameter vector, projections and reprojection errors equal the reference's, and bundle_adjust keeps the object classes and lowers
  the reference's initial cost."""
  import numpy as np
  from conftest import load_golden
  from multical_b200.calibration import from_scene
  from multical_b200.motion import HandEye, RollingFrames
  from multical_b200.pose_set import pose_table
  scene, z = load_golden("refcalib_" + motion)
  calib = from_scene(scene)
  if motion == "rolling":
    calib = calib.copy(motion=RollingFrames(z["frame_poses"], z["frame_poses_end"], z["frame_valid"], [str(i) for i in range(scene["F"])]))
  elif motion == "hand_eye":
    calib = calib.copy(motion=HandEye(pose_table(z["base_wrt_gripper"], z["frame_valid"]), z["world_wrt_base"], z["gripper_wrt_camera"]))
  calib = calib.enable(camera_poses=False, cameras=False) if motion == "hand_eye" else calib.enable(cameras=True)
  assert np.abs(np.asarray(calib.param_vec) - z["x0"]).max() < 1e-12
  assert np.abs(np.asarray(calib.reprojected.points)[z["ok"]] - z["reprojected"]).max() < 1e-9
  assert np.abs(np.asarray(calib.reprojection_error) - z["reprojection_error"]).max() < 1e-9
  out = calib.bundle_adjust(max_iterations=10)
  assert type(out.motion) is type(calib.motion) and type(out.cameras[0]) is type(calib.cameras[0])
  r = (np.asarray(out.reprojected.points) - np.asarray(out.point_table.points))[np.asarray(out.inliers)]
  assert abs(0.5 * float(np.sum(r ** 2)) - out.last_solve.cost) <= 1e-9 * out.last_solve.cost
  assert out.last_solve.cost < float(z["cost0"])


def test_cfg1_the_reference_cpu_case_end_to_end():
  """BASELINE.json configs[0] (2 cameras x 20 frames of charuco_16x22, ~5k corners: the case the reference itself runs on the CPU):
  Calibration.bundle_adjust through the C-ABI against the reference algorithm (oracle: dense numpy evaluate + the identical scipy call)."""
  import numpy as np
  from multical_b200 import synthetic
  from multical_b200.calibration import from_scene
  from oracle.ba_oracle import Problem
  scene = synthetic.make_workload("cfg1")
  calib = from_scene(scene).enable(cameras=True)
  prob = Problem.from_scene(scene, optimize=dict(cameras=True))
  assert np.array_equal(calib.param_vec, prob.param_vec)                                   # indexing / layout: bit exact
  eng = calib._upload(calib.inliers)
  assert 4000 < eng.N < 8000 and np.abs(eng.residuals() - prob.residuals()).max() < 1e-9
  out = calib.bundle_adjust()
  _, ref = prob.bundle_adjust()
  assert out.last_solve.cost <= ref.cost * (1 + 1e-6) and out.last_solve.nfev <= ref.nfev
  rms = np.sqrt(np.mean(out.reprojection_error ** 2))
  assert abs(rms - np.sqrt(2 * ref.cost / eng.N)) < 1e-3 and 0.3 < rms < 0.5              # 0.3 px noise per coordinate
