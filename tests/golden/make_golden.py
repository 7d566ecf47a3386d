"""Generate golden vectors from the UNMODIFIED reference (imported through tests/refshim).

Run in the build container only (`/root/reference` must exist):
    python tests/golden/make_golden.py
For each small synthetic scene it stores the inputs (plain arrays) and what the reference computes:
  x0            Calibration.param_vec                          (parameters.py:44-46)
  r0, r1        evaluate(x0), evaluate(x1)                     (calibration.py:204-206)
  sp_indptr/sp_indices   Calibration.sparsity_matrix (CSR)     (calibration.py:173-196)
  err_valid     Calibration.reprojection_error                 (calibration.py:134-136)
  ba_x, ba_cost, ba_nfev, ba_rms   bundle_adjust() result      (calibration.py:199-212)
The bundle_adjust trajectory of the reference is numerically chaotic (LSMR inner solves on a gauge-
singular Jacobian: a 1e-13 px perturbation of the residuals changes the final cost in the 5th digit,
see DESIGN.md), so ba_* are compared with a tolerance that reflects that, not bit-wise.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "refshim"))

from multical_b200 import synthetic  # noqa: E402
import loader  # noqa: E402

CASES = {
  "standard_2x6": dict(C=2, F=6, vis=0.5, seed=11, model="standard"),
  "fisheye_3x5": dict(C=3, F=5, vis=0.5, seed=12, model="fisheye"),
  "rational_2x5": dict(C=2, F=5, vis=0.5, seed=13, model="rational"),
  "cube3_3x6": dict(C=3, F=6, vis=0.6, seed=14, model="standard", boards=("cube", 10, 10, 0.04, 3), rig="dome"),
  "poses_only_2x6": dict(C=2, F=6, vis=0.5, seed=15, model="standard"),
  "invalid_poses_3x6": dict(C=3, F=6, vis=0.5, seed=16, model="standard"),
  "thin_prism_2x5": dict(C=2, F=5, vis=0.5, seed=17, model="thin_prism"),
  "tilted_2x5": dict(C=2, F=5, vis=0.5, seed=18, model="tilted"),
}


def outlier_case(ref, name="outliers_3x6"):
  """The steps either side of bundle_adjust, from the running reference, at a state where rejection means something (true
  parameters, 0.3 px noise, 2 % gross outliers):
    thr_q75x5       select_threshold(0.75, 5.0)(calib.reprojection_error)              (calibration.py:37-40)
    inliers_thr     calib.reject_outliers(thr_q75x5).inliers                           (calibration.py:240-252)
    inliers_q95     calib.reject_outliers_quantile(0.95).inliers                       (calibration.py:234-238)
    adj_inliers, adj_rms   calib.adjust_outliers(2, select_outliers=select_threshold(0.75, 5.0)) -> inlier mask and the
                    RMS error of its inliers                                           (calibration.py:254-268)"""
  scene = synthetic.make_scene(C=3, F=6, vis=0.5, seed=19, model="standard", outlier_fraction=0.02)
  calib = loader.build_calibration(ref, scene, guess=False).enable(cameras=True)
  err = calib.reprojection_error
  thr = ref.select_threshold(quantile=0.75, factor=5.0)(err)
  adjusted = calib.adjust_outliers(num_adjustments=2, select_outliers=ref.select_threshold(quantile=0.75, factor=5.0))
  gt = scene["gt"]
  data = dict(
    model=scene["model"], points=scene["points"], valid=scene["valid"],
    cam_valid=scene["cam_valid"], frame_valid=scene["frame_valid"], board_valid=scene["board_valid"],
    board_points=np.stack(scene["board_points"]), K=gt["K"], dist=gt["dist"],
    cam_poses=gt["cam_poses"], frame_poses=gt["frame_poses"], board_poses=gt["board_poses"],
    image_size=np.array(scene["image_size"]), cameras_enabled=True,
    x0=calib.param_vec, err_valid=err, thr_q75x5=float(thr),
    inliers_thr=calib.reject_outliers(thr).inliers, inliers_q95=calib.reject_outliers_quantile(0.95).inliers,
    adj_inliers=adjusted.inliers, adj_rms=float(np.sqrt(np.mean(adjusted.reprojection_inliers ** 2))))
  path = os.path.join(HERE, name + ".npz")
  np.savez_compressed(path, **data)
  print(name, "valid", int(calib.valid.sum()), "thr", thr, "kept", int(data["inliers_thr"].sum()), "q95 kept",
        int(data["inliers_q95"].sum()), "adjusted kept", int(data["adj_inliers"].sum()), "rms", data["adj_rms"],
        os.path.getsize(path) // 1024, "KB")


def small_motion(rng, n, rot=0.01, trans=0.01):
  from scipy.spatial.transform import Rotation
  T = np.tile(np.eye(4), (n, 1, 1))
  T[:, :3, :3] = Rotation.from_rotvec(rng.normal(0, rot, (n, 3))).as_matrix()
  T[:, :3, 3] = rng.normal(0, trans, (n, 3))
  return T


def motion_cases(ref, only):
  """The two motion models the BASELINE configurations do not use (SURVEY.md §8f rank 2), pinned the same way as the static
  cases: parameter layout, evaluate() at two points, Jacobian sparsity, per-corner error, one bundle_adjust of the reference.
    rolling_2x6   RollingFrames: start pose = the scene's frame pose, end pose = start moved by ~1 cm / 0.6 deg; the blend
                  weight of a corner is its observed row / image height           (motion/rolling_frames.py:15-41,66-150)
    handeye_2x6   HandEye: frame pose = gripper_wrt_camera @ base_wrt_gripper[f] @ world_wrt_base; arm poses constructed so that
                  the scene's frame poses are reproduced exactly, then the two optimised transforms are perturbed; blocks enabled
                  as HandEyeCalibration.initialise leaves them (optimization/hand_eye.py:37)   (motion/hand_eye.py:14-90)"""
  for name in ("rolling_2x6", "handeye_2x6"):
    rng = np.random.default_rng(200)       # per case: a fixture does not depend on which other cases are regenerated with it
    if only and name not in only: continue
    scene = synthetic.make_scene(C=2, F=6, vis=0.5, seed=20 if name.startswith("rolling") else 21, model="standard")
    # hand-eye fixes cameras and camera poses (optimization/hand_eye.py:37), so that case starts from their true values
    src = scene["init"] if name.startswith("rolling") else scene["gt"]
    extra = {}
    if name.startswith("rolling"):
      end = small_motion(rng, scene["F"]) @ src["frame_poses"]
      calib = loader.build_calibration(ref, scene, motion=("rolling", end)).enable(cameras=True)
      extra = dict(motion="rolling", frame_poses_end=end)
      enabled = dict(cameras=True)
    else:
      g2c = small_motion(rng, 1, 0.3, 0.1)[0]; w2b = small_motion(rng, 1, 0.5, 0.5)[0]
      arm = np.linalg.inv(g2c)[None] @ src["frame_poses"] @ np.linalg.inv(w2b)[None]        # base_wrt_gripper per frame
      g2c0 = small_motion(rng, 1, 0.005, 0.005)[0] @ g2c; w2b0 = w2b @ small_motion(rng, 1, 0.005, 0.005)[0]
      calib = loader.build_calibration(ref, scene, guess=False, motion=("hand_eye", arm, w2b0, g2c0)).enable(camera_poses=False, cameras=False)
      extra = dict(motion="hand_eye", base_wrt_gripper=arm, world_wrt_base=w2b0, gripper_wrt_camera=g2c0)
      enabled = dict(camera_poses=False, cameras=False)
    x0 = calib.param_vec
    inl = calib.inliers
    def evaluate(x):
      c = calib.with_param_vec(x)
      return (c.reprojected.points - c.point_table.points)[inl].ravel()
    x1 = x0 + np.random.default_rng(101).normal(0, 1e-3, x0.size)
    S = calib.sparsity_matrix.tocsr(); S.sort_indices()
    out = calib.bundle_adjust()
    data = dict(
      model=scene["model"], points=scene["points"], valid=scene["valid"],
      cam_valid=scene["cam_valid"], frame_valid=scene["frame_valid"], board_valid=scene["board_valid"],
      board_points=np.stack(scene["board_points"]), K=src["K"], dist=src["dist"],
      cam_poses=src["cam_poses"], frame_poses=src["frame_poses"], board_poses=src["board_poses"],
      image_size=np.array(scene["image_size"]),
      enabled_keys=np.array(list(enabled.keys())), enabled_values=np.array(list(enabled.values())),
      x0=x0, x1=x1, r0=evaluate(x0), r1=evaluate(x1), sp_indptr=S.indptr, sp_indices=S.indices, sp_shape=np.array(S.shape),
      err_valid=calib.reprojection_error, ba_x=out.param_vec,
      ba_cost=0.5 * float(np.sum(evaluate(out.param_vec) ** 2)),
      ba_rms=float(np.sqrt(np.mean(out.reprojection_error ** 2))), **extra)
    # the same model with boards=True (board points as parameters, board/charuco.py:112-117): layout and evaluate() at two points
    cb = calib.enable(boards=True)
    xb0 = cb.param_vec
    xb1 = xb0 + np.random.default_rng(102).normal(0, 1e-4, xb0.size)
    def evaluate_b(x):
      c = cb.with_param_vec(x)
      return (c.reprojected.points - c.point_table.points)[inl].ravel()
    data.update(boards_x0=xb0, boards_x1=xb1, boards_r1=evaluate_b(xb1))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **data)
    print(name, "N", int(inl.sum()), "n", x0.size, "cost0", 0.5 * float(np.sum(data["r0"] ** 2)), "cost", data["ba_cost"],
          "rms", data["ba_rms"], os.path.getsize(path) // 1024, "KB")


def pnp_cases(ref, only):
  """Board-pose initialisation (SURVEY.md §8f rank 4): the reference's own tables.make_pose_table (tables.py:44-66) -> extract_pose ->
  board.estimate_pose_points (board/common.py:36-47) on synthetic detections, with boards that answer `has_min_detections` through the
  reference's has_min_detections_grid (board/common.py:30-34) exactly as CharucoBoard does (charuco.py:104-109; min_rows=3, min_points=20).
    pnp_std_3x6      pinhole 5-coefficient cameras, sparse views (some below the minimum -> invalid_pose), 0.3 px noise
    pnp_fisheye_2x5  fisheye cameras (camera_fisheye.py:108-111 undistortion)
    pnp_cube_3x4     three 10x10 boards per frame, exclude_bad_poses with a limit that rejects part of the views"""
  from multical.board.common import estimate_pose_points, has_min_detections_grid
  from multical import tables

  class GridBoard(ref.SyntheticBoard):
    def __init__(self, adjusted_points, size, min_points=20, min_rows=3):
      super().__init__(adjusted_points); self.size, self.min_points, self.min_rows = size, min_points, min_rows
    def has_min_detections(self, detections):
      return has_min_detections_grid(self.size, detections.ids, min_points=self.min_points, min_rows=self.min_rows)
    def estimate_pose_points(self, camera, detections):
      return estimate_pose_points(self, camera, detections)

  cases = {
    "pnp_std_3x6": (dict(C=3, F=6, vis=0.08, seed=31, model="standard"), (16, 22), dict()),
    "pnp_fisheye_2x5": (dict(C=2, F=5, vis=0.3, seed=32, model="fisheye"), (16, 22), dict()),
    "pnp_cube_3x4": (dict(C=3, F=4, vis=0.5, seed=33, model="standard", boards=("cube", 10, 10, 0.04, 3), rig="dome"), (10, 10),
                     dict(exclude_bad_poses=True, pose_error_limit=0.305)),
  }
  for name, (kw, size, opts) in cases.items():
    if only and name not in only: continue
    scene = synthetic.make_scene(**kw)
    calib = loader.build_calibration(ref, scene, guess=False)
    boards = [GridBoard(p, size) for p in scene["board_points"]]
    table = tables.make_pose_table(calib.point_table, boards, calib.cameras, opts.get("exclude_bad_poses", False), opts.get("pose_error_limit", 1.0))
    data = dict(model=scene["model"], points=scene["points"], valid=scene["valid"], board_points=np.stack(scene["board_points"]),
                K=scene["gt"]["K"], dist=scene["gt"]["dist"], image_size=np.array(scene["image_size"]), grid=np.array([*size, 1, 20, 3]),
                exclude_bad_poses=bool(opts.get("exclude_bad_poses", False)), pose_error_limit=float(opts.get("pose_error_limit", 1.0)),
                poses=table.poses, pose_valid=table.valid, num_points=table.num_points, reprojection_error=table.reprojection_error,
                view_angles=table.view_angles)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **data)
    print(name, "views", table.valid.size, "valid", int(table.valid.sum()), "max err", float(np.max(table.reprojection_error)), os.path.getsize(path) // 1024, "KB")


def scene_arrays(scene, src):
  """The inputs of a scene in the layout tests/conftest.py load_golden reads (src: the scene's "init" or "gt" estimates)."""
  return dict(model=scene["model"], points=scene["points"], valid=scene["valid"],
              cam_valid=scene["cam_valid"], frame_valid=scene["frame_valid"], board_valid=scene["board_valid"],
              board_points=np.stack(scene["board_points"]), K=src["K"], dist=src["dist"],
              cam_poses=src["cam_poses"], frame_poses=src["frame_poses"], board_poses=src["board_poses"],
              image_size=np.array(scene["image_size"]))


def dome_case(ref, name="dome_cube2_3x5"):
  """Three cameras on a dome around two 10x10 cube faces (tests/test_oracle.py test_oracle_against_reference_dome_rig):
    x0            Calibration.param_vec
    x1, r1        a perturbed parameter vector and the reference's residuals there
    sp_*          Calibration.sparsity_matrix (CSR, sorted indices, with its values)"""
  scene = synthetic.make_scene(C=3, F=5, vis=0.6, seed=21, boards=("cube", 10, 10, 0.04, 2), rig="dome")
  calib = loader.build_calibration(ref, scene).enable(cameras=True)
  x0 = calib.param_vec
  x1 = x0 + np.random.default_rng(5).normal(0, 1e-3, x0.size)
  c1 = calib.with_param_vec(x1)
  r1 = (c1.reprojected.points - c1.point_table.points)[calib.inliers].ravel()
  S = calib.sparsity_matrix.tocsr(); S.sort_indices()
  data = dict(scene_arrays(scene, scene["init"]), cameras_enabled=True, x0=x0, x1=x1, r1=r1,
              sp_indptr=S.indptr, sp_indices=S.indices, sp_data=S.data, sp_shape=np.array(S.shape))
  path = os.path.join(HERE, name + ".npz")
  np.savez_compressed(path, **data)
  print(name, "N", int(calib.inliers.sum()), "n", x0.size, os.path.getsize(path) // 1024, "KB")


def reference_calibration_cases(ref, only):
  """What tests/test_simt_kernels.py test_calibration_over_the_reference_objects compares this package's Calibration against, for
  the static, rolling and hand-eye motion models of one small scene (the motion inputs are stored beside the scene):
    x0                   Calibration.param_vec
    ok, reprojected      reprojected.valid & point_table.valid, and reprojected.points where it holds
    reprojection_error   Calibration.reprojection_error
    cost0                half the squared inlier residuals at x0"""
  for motion in ("static", "rolling", "hand_eye"):
    name = "refcalib_" + motion
    if only and name not in only: continue
    scene = synthetic.make_scene(C=2, F=5, vis=0.4, seed=77)
    spec, extra = None, {}
    if motion == "rolling":
      end = scene["init"]["frame_poses"].copy(); end[:, :3, 3] += 0.005
      spec, extra = ("rolling", end), dict(frame_poses_end=end)
    elif motion == "hand_eye":
      spec = ("hand_eye", scene["init"]["frame_poses"], np.eye(4), np.eye(4))          # arm poses = frame estimates, identity hand-eye pair
      extra = dict(base_wrt_gripper=spec[1], world_wrt_base=spec[2], gripper_wrt_camera=spec[3])
    rc = loader.build_calibration(ref, scene, motion=spec)
    rc = rc.enable(camera_poses=False, cameras=False) if motion == "hand_eye" else rc.enable(cameras=True)
    ok = np.asarray(rc.reprojected.valid) & np.asarray(rc.point_table.valid)
    r0 = (np.asarray(rc.reprojected.points) - np.asarray(rc.point_table.points))[np.asarray(rc.inliers)]
    data = dict(scene_arrays(scene, scene["init"]), motion=motion, x0=np.asarray(rc.param_vec), ok=ok,
                reprojected=np.asarray(rc.reprojected.points)[ok], reprojection_error=np.asarray(rc.reprojection_error),
                cost0=0.5 * float(np.sum(r0 ** 2)), **extra)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **data)
    print(name, "n", data["x0"].size, "ok", int(ok.sum()), "cost0", data["cost0"], os.path.getsize(path) // 1024, "KB")


def main():
  ref = loader.load()
  only = sys.argv[1:]          # optional: regenerate just the named cases (existing fixtures stay byte-identical)
  if not only or "dome_cube2_3x5" in only: dome_case(ref)
  if not only or any(n.startswith("refcalib_") for n in only): reference_calibration_cases(ref, only)
  if not only or "outliers_3x6" in only: outlier_case(ref)
  if not only or any(n in only for n in ("rolling_2x6", "handeye_2x6")): motion_cases(ref, only)
  if not only or any(n.startswith("pnp_") for n in only): pnp_cases(ref, only)
  for name, kw in CASES.items():
    if only and name not in only: continue
    scene = synthetic.make_scene(**kw)
    if name.startswith("invalid"):
      scene["frame_valid"][2] = False
      scene["cam_valid"][1] = False
    calib = loader.build_calibration(ref, scene)
    if not name.startswith("poses_only"):
      calib = calib.enable(cameras=True)
    x0 = calib.param_vec
    inl = calib.inliers
    def evaluate(x):
      c = calib.with_param_vec(x)
      return (c.reprojected.points - c.point_table.points)[inl].ravel()
    rng = np.random.default_rng(100)
    x1 = x0 + rng.normal(0, 1e-3, x0.size)
    S = calib.sparsity_matrix.tocsr(); S.sort_indices()
    out = calib.bundle_adjust()
    data = dict(
      model=scene["model"], points=scene["points"], valid=scene["valid"],
      cam_valid=scene["cam_valid"], frame_valid=scene["frame_valid"], board_valid=scene["board_valid"],
      board_points=np.stack(scene["board_points"]), K=scene["init"]["K"], dist=scene["init"]["dist"],
      cam_poses=scene["init"]["cam_poses"], frame_poses=scene["init"]["frame_poses"], board_poses=scene["init"]["board_poses"],
      image_size=np.array(scene["image_size"]), cameras_enabled=not name.startswith("poses_only"),
      x0=x0, x1=x1, r0=evaluate(x0), r1=evaluate(x1), sp_indptr=S.indptr, sp_indices=S.indices, sp_shape=np.array(S.shape),
      err_valid=calib.reprojection_error, ba_x=out.param_vec,
      ba_cost=0.5 * float(np.sum(evaluate(out.param_vec) ** 2)),
      ba_rms=float(np.sqrt(np.mean(out.reprojection_error ** 2))))
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **data)
    print(name, "N", int(inl.sum()), "n", x0.size, "cost", data["ba_cost"], "rms", data["ba_rms"], os.path.getsize(path) // 1024, "KB")


if __name__ == "__main__":
  main()
