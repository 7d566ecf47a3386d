"""CPU: the oracle (oracle/ba_oracle.py) against the golden vectors produced by the running reference
(tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import GOLDEN_CASES, ROOT, load_golden, optimize_of
from oracle.ba_oracle import Problem


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_matches_golden_vectors(name):
  scene, z = load_golden(name)
  prob = Problem.from_scene(scene, optimize=optimize_of(z))
  # parameter vector layout: bit exact (parameters.py:104-106)
  assert np.array_equal(prob.param_vec, z["x0"])
  # evaluate() at two points (calibration.py:204-206): fp64, same formulas -> 1e-9 px bar, observed ~1e-13
  assert np.abs(prob.residuals() - z["r0"]).max() < 1e-9
  assert np.abs(prob.residuals(z["x1"]) - z["r1"]).max() < 1e-9
  # Jacobian sparsity pattern: exact
  S = prob.sparsity_matrix().tocsr(); S.sort_indices()
  assert tuple(S.shape) == tuple(z["sp_shape"])
  assert np.array_equal(S.indptr, z["sp_indptr"]) and np.array_equal(S.indices, z["sp_indices"])
  # per-corner reprojection error over valid (calibration.py:134-136)
  err, mask = prob.reprojection_error()
  assert np.abs(err[mask] - z["err_valid"]).max() < 1e-9


def test_oracle_outlier_steps_match_reference_golden():
  """reprojection_error / select_threshold / reject_outliers / reject_outliers_quantile of the running reference
  (tests/golden/make_golden.py outlier_case; calibration.py:37-40, 234-252)."""
  scene, z = load_golden("outliers_3x6")
  prob = Problem.from_scene(scene, optimize=dict(cameras=True))
  assert np.array_equal(prob.param_vec, z["x0"])
  err, mask = prob.reprojection_error()
  assert np.abs(err[mask] - z["err_valid"]).max() < 1e-9
  thr = np.quantile(err[mask], 0.75) * 5.0
  assert abs(thr - float(z["thr_q75x5"])) < 1e-9
  assert np.array_equal((err < float(z["thr_q75x5"])) & mask, z["inliers_thr"])
  assert np.array_equal((err < np.quantile(err[mask], 0.95)) & mask, z["inliers_q95"])
  assert z["inliers_thr"].sum() < mask.sum() and np.array_equal(z["adj_inliers"] & mask, z["adj_inliers"])


def motion_problem(name):
  scene, z = load_golden(name)
  kw = dict(optimize=dict(zip((str(k) for k in z["enabled_keys"]), (bool(v) for v in z["enabled_values"]))),
            motion=str(z["motion"]), image_size=z["image_size"])
  for key in ("frame_poses_end", "base_wrt_gripper", "world_wrt_base", "gripper_wrt_camera"):
    if key in z: kw[key] = z[key]
  return Problem.from_scene(scene, **kw), z


@pytest.mark.parametrize("name", ["rolling_2x6", "handeye_2x6"])
def test_oracle_motion_models_match_reference_golden(name):
  """RollingFrames (motion/rolling_frames.py) and HandEye (motion/hand_eye.py) -- SURVEY.md §8f rank 2, not yet on the GPU
  path; the restatement is pinned now so that the device work has an oracle to be checked against."""
  prob, z = motion_problem(name)
  assert np.array_equal(prob.param_vec, z["x0"])                         # block order and the motion block's own layout
  assert np.abs(prob.residuals() - z["r0"]).max() < 1e-9
  assert np.abs(prob.residuals(z["x1"]) - z["r1"]).max() < 1e-9          # x1 moves start/end (or the two hand-eye transforms) apart
  S = prob.sparsity_matrix().tocsr(); S.sort_indices()
  assert tuple(S.shape) == tuple(z["sp_shape"])
  assert np.array_equal(S.indptr, z["sp_indptr"]) and np.array_equal(S.indices, z["sp_indices"])
  err, mask = prob.reprojection_error()
  assert np.abs(err[mask] - z["err_valid"]).max() < 1e-9
  pb = prob.copy(optimize=dict(prob.optimize, boards=True))             # boards=True under the same motion model
  assert np.abs(pb.param_vec - z["boards_x0"]).max() < 1e-12 and np.abs(pb.residuals(z["boards_x1"]) - z["boards_r1"]).max() < 1e-9
  out, res = prob.bundle_adjust()
  assert abs(res.cost - float(z["ba_cost"])) / float(z["ba_cost"]) < 1e-3
  e2, m2 = out.reprojection_error()
  assert abs(np.sqrt(np.mean(e2[m2] ** 2)) - float(z["ba_rms"])) < 1e-2


@pytest.mark.parametrize("name", ["pnp_std_3x6", "pnp_fisheye_2x5", "pnp_cube_3x4"])
def test_pnp_oracle_matches_reference_golden(name):
  """oracle/pnp_oracle.py (board/common.py:30-47 + tables.py:34-66 restated over cv2) against the reference's own make_pose_table."""
  from oracle import pnp_oracle
  z = dict(np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"), allow_pickle=False))
  grid = tuple(int(v) for v in z["grid"])
  poses, ok, npts, err = pnp_oracle.make_pose_table(str(z["model"]), z["K"], z["dist"], z["board_points"], [grid] * z["board_points"].shape[0],
                                                    z["points"], z["valid"], bool(z["exclude_bad_poses"]), float(z["pose_error_limit"]))
  assert np.array_equal(ok, z["pose_valid"]) and np.array_equal(npts, z["num_points"])
  assert np.abs(poses - z["poses"]).max() < 1e-12 and np.abs(err - z["reprojection_error"]).max() < 1e-12   # same OpenCV calls


@pytest.mark.parametrize("name", ["standard_2x6", "cube3_3x6"])
def test_oracle_bundle_adjust_close_to_reference_run(name):
  """The reference's TRF+LSMR trajectory is chaotic at the 1e-5 level in final cost (DESIGN.md), so the
  restated solve is only required to land within the reference's own ftol (1e-4) of its final cost."""
  scene, z = load_golden(name)
  prob = Problem.from_scene(scene, optimize=optimize_of(z))
  out, res = prob.bundle_adjust()
  assert abs(res.cost - float(z["ba_cost"])) / float(z["ba_cost"]) < 1e-3
  err, mask = out.reprojection_error()
  assert abs(np.sqrt(np.mean(err[mask] ** 2)) - float(z["ba_rms"])) < 1e-2


def test_oracle_against_reference_dome_rig():
  """Three cameras on a dome around two cube faces: parameter layout, residuals at a perturbed point and the Jacobian sparsity
  (pattern and values) against what the reference computed (tests/golden/make_golden.py dome_case)."""
  scene, z = load_golden("dome_cube2_3x5")
  prob = Problem.from_scene(scene, optimize=optimize_of(z))
  assert np.array_equal(z["x0"], prob.param_vec)
  assert np.abs(z["r1"] - prob.residuals(z["x1"])).max() < 1e-9
  S = sp.csr_matrix((z["sp_data"], z["sp_indices"], z["sp_indptr"]), shape=tuple(z["sp_shape"]))
  assert (S != prob.sparsity_matrix()).nnz == 0
