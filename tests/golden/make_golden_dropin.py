"""Goldens of the drop-in test (tests/test_dropin_reference.py), produced by the unmodified reference under
oracle/ref_shims.py:

* the reference's own `SLAM.init()` / `SLAM.process_next_frame()` loop (slam/slam.py:81-166) -- CV initialisation,
  the GridSample(0.4) -> ToTensor preprocessing chain, `icp_F2M` with a kd-tree map of 4 frames and 6 fixed
  point-to-plane GN alignments -- on six 32x512 synthetic scans: per frame the data_dict's keys, `init_rpose`,
  `sample_indices`, `odometry_pose` and the shape of `odometry_pc`, plus the shape of `get_relative_poses()`;
* the values of config/slam/odometry/icp_odometry.yaml and the defaults of `ICPFrameToModelConfig`;
* the error each alignment raises when handed a `mask`.

    python tests/golden/make_golden_dropin.py        (needs a reference checkout, PLS_REFERENCE_ROOT)  ->  dropin_reference.npz
"""
import dataclasses
import json
import os
import sys

import numpy as np
import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_shims  # noqa: E402
from pylidar_slam_b200 import synthetic as syn  # noqa: E402

ref_shims.install()
import slam.common.pose as pose  # noqa: E402
import slam.common.projection as projection  # noqa: E402
import slam.initialization as initialization  # noqa: E402
import slam.odometry.alignment as alignment  # noqa: E402
import slam.odometry.icp_odometry as icp  # noqa: E402
import slam.odometry.local_map as local_map  # noqa: E402
import slam.preprocessing as preprocessing  # noqa: E402
import slam.slam as slam  # noqa: E402

H, W, VOXEL, FRAMES = 32, 512, 0.4, 6
torch.set_num_threads(1)  # the reference's z-buffer scatter is racy with more (DESIGN.md section 2)


def slam_loop():
    cfg = slam.SLAMConfig(
        initialization=initialization.CVConfig(),
        preprocessing=preprocessing.PreprocessingConfig(filters={
            "2": dict(filter_name="grid_sample", voxel_size=VOXEL, pointcloud_key="numpy_pc"),
            "3": dict(filter_name="to_tensor", keys=dict(sample_points="input_data"))}),
        odometry=icp.ICPFrameToModelConfig(
            algorithm="icp_F2M", data_key="input_data", max_num_alignments=6, threshold_delta_pose=0.0,
            local_map=local_map.KdTreeLocalMapConfig(local_map_size=4),
            alignment=alignment.GaussNewtonPointToPlaneConfig(
                gauss_newton_config=dict(scheme="geman_mcclure", sigma=0.3, max_iters=1))))
    projector = projection.SphericalProjector(height=H, width=W, up_fov=3.0, down_fov=-24.0)
    algo = slam.SLAM(cfg, projector=projector, pose=pose.Pose("euler"), device=torch.device("cpu"), viz_num_pointclouds=1)
    algo.init()
    out, keys = {}, []
    for k in range(FRAMES):
        dd = {"numpy_pc": syn.scan(k, H, W)}
        algo.process_next_frame(dd)
        keys.append(sorted(dd.keys()))
        out[f"init_rpose_{k}"] = np.asarray(dd["init_rpose"], dtype=np.float64)
        out[f"sample_indices_{k}"] = np.asarray(dd["sample_indices"])
        if "odometry_pose" in dd:
            out[f"odometry_pose_{k}"] = dd["odometry_pose"]
            out[f"odometry_pc_shape_{k}"] = np.asarray(dd["odometry_pc"].shape, dtype=np.int64)
    out["relative_poses_shape"] = np.asarray(algo.odometry.get_relative_poses().shape, dtype=np.int64)
    return out, keys


def mask_errors():
    n = 128
    rs = np.random.RandomState(3)
    pts = torch.from_numpy(rs.randn(1, n, 3).astype(np.float32))
    nrm = torch.nn.functional.normalize(torch.from_numpy(rs.randn(1, n, 3).astype(np.float32)), dim=2)
    mask = torch.ones(1, n, 1)
    gn = dict(scheme="geman_mcclure", sigma=0.3, max_iters=1)
    plane = alignment.GaussNewtonPointToPlaneAlignment(alignment.GaussNewtonPointToPlaneConfig(gauss_newton_config=gn),
                                                       pose=pose.Pose("euler"))
    point = alignment.GaussNewtonPointToPointAlignment(alignment.GNPointToPointConfig(gauss_newton_config=gn),
                                                       pose=pose.Pose("euler"))
    errors = {}
    for name, call in (("point_to_plane", lambda: plane.align(pts, pts + 0.01, nrm, mask=mask)),
                       ("point_to_point", lambda: point.align(pts, pts + 0.01, mask=mask))):
        try:
            call()
            errors[name] = None
        except Exception as e:
            errors[name] = {"type": type(e).__name__, "message": str(e)}
    return errors


def main():
    out, keys = slam_loop()
    with open(os.path.join(ref_shims.REFERENCE_ROOT, "config", "slam", "odometry", "icp_odometry.yaml")) as fh:
        icp_yaml = yaml.safe_load(fh)
    defaults = {f.name: f.default for f in dataclasses.fields(icp.ICPFrameToModelConfig)
                if isinstance(f.default, (str, int, float, bool))}
    meta = {"frames": FRAMES, "keys": keys, "icp_odometry_yaml": icp_yaml, "config_defaults": defaults,
            "mask_errors": mask_errors()}
    out["meta"] = np.array(json.dumps(meta, sort_keys=True))
    np.savez_compressed(os.path.join(HERE, "dropin_reference.npz"), **out)
    print("wrote", os.path.join(HERE, "dropin_reference.npz"), sorted(out))


if __name__ == "__main__":
    main()
