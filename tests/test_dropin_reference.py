"""The drop-in claim: run in pyLiDAR-SLAM's SLAM loop, `pylidar_slam_b200.ICPFrameToModel` hands the caller what the
reference's own `icp_F2M` hands it.  tests/golden/make_golden_dropin.py ran the UNMODIFIED reference's
`SLAM.init()` / `SLAM.process_next_frame()` loop on six synthetic scans and stored what a caller reads from it
(tests/golden/dropin_reference.npz).  Here the same loop -- slam/slam.py:118-140 with a constant-velocity
initialisation and no loop closure or backend: `init_rpose` = the last relative pose, the GridSample -> ToTensor
preprocessing chain, the odometry, `save_real_motion` -- drives this package's classes, constructed with the kwargs
the reference's `ODOMETRY.load(config.odometry, projector=, pose=, device=, ...)` passes.  No GPU here: the classes run
on the test-only CPU stand-in for the C ABI (tests/dryrun_next_rows.FakeContext, oracle arithmetic), so what is
checked is everything ABOVE the C ABI: registry and config plumbing, constructor kwargs, data_dict keys in and out,
the pose bookkeeping the caller reads -- against the reference's own `icp_F2M` on the same frames."""
import json
import os
import sys
import types
from enum import Enum

import numpy as np
import pytest
import torch
import yaml

import dryrun_next_rows as dry
from conftest import GOLDEN, pose_errors
from pylidar_slam_b200 import synthetic as syn

H, W, VOXEL, FRAMES = 32, 512, 0.4, 6


@pytest.fixture(scope="module")
def golden():
    g = np.load(os.path.join(GOLDEN, "dropin_reference.npz"))
    return g, json.loads(str(g["meta"]))


@pytest.fixture
def b200(monkeypatch):
    import pylidar_slam_b200 as pkg
    from pylidar_slam_b200 import _lib, common
    monkeypatch.setattr(_lib, "Context", dry.FakeContext)          # CPU stand-in for the C ABI (tests only)
    monkeypatch.setattr(common, "_default_ctx", dry.FakeContext())
    return pkg


def _odometry_config(b200, **kwargs):
    return b200.ICPFrameToModelConfig(
        algorithm="icp_F2M_b200", data_key="input_data", max_num_alignments=6, threshold_delta_pose=0.0,
        local_map=b200.KdTreeLocalMapConfig(local_map_size=4),
        alignment=b200.GaussNewtonPointToPlaneConfig(gauss_newton_config=dict(scheme="geman_mcclure", sigma=0.3, max_iters=1)),
        **kwargs)


def _loader_kwargs(b200):
    """What SLAM.init hands ODOMETRY.load besides the config.  A CPU box has no cuda device to hand to torch: the
    odometry is told cuda:0 (a string; the stand-in backend never touches a device)."""
    return dict(projector=b200.SphericalProjector(height=H, width=W, up_fov=3.0, down_fov=-24.0), pose=b200.Pose("euler"),
                device="cuda:0", viz_num_pointclouds=1)


def _run(b200):
    preprocessing = b200.Preprocessing(b200.PreprocessingConfig(filters={
        "2": dict(filter_name="grid_sample", voxel_size=VOXEL, pointcloud_key="numpy_pc"),
        "3": dict(filter_name="to_tensor", keys=dict(sample_points="input_data"))}), device=torch.device("cpu"))
    odometry = b200.ICPFrameToModel(_odometry_config(b200), **_loader_kwargs(b200))
    odometry.init()
    initial_estimate, frames = np.eye(4), []                          # ConstantVelocityInitialization.init
    for k in range(FRAMES):
        data_dict = {"numpy_pc": syn.scan(k, H, W)}
        data_dict["init_rpose"] = initial_estimate                    # initialization.next_frame
        preprocessing.forward(data_dict)
        odometry.process_next_frame(data_dict)
        if odometry.relative_pose_key() in data_dict:
            initial_estimate = data_dict[odometry.relative_pose_key()]  # initialization.save_real_motion
        frames.append(data_dict)
    return odometry, frames


def test_b200_odometry_drops_into_the_reference_slam_loop(b200, golden):
    g, meta = golden
    threads = torch.get_num_threads()
    torch.set_num_threads(1)  # the z-buffer scatter of the oracle arithmetic is racy with more (DESIGN.md section 2)
    try:
        ours, frames = _run(b200)
    finally:
        torch.set_num_threads(threads)
    assert len(meta["keys"]) == FRAMES
    for k, b in enumerate(frames):
        assert sorted(b.keys()) == meta["keys"][k], (k, sorted(b.keys()), meta["keys"][k])
        np.testing.assert_array_equal(b["sample_indices"], g[f"sample_indices_{k}"])
        if k == 0:
            assert "odometry_pose" not in b  # the first frame only initialises the map (icp_odometry.py:171-181)
            continue
        assert b["odometry_pose"].shape == (4, 4) and b["odometry_pose"].dtype == np.float32
        assert b["odometry_pc"].shape == tuple(g[f"odometry_pc_shape_{k}"])
        dt, ang = pose_errors(b["odometry_pose"], g[f"odometry_pose_{k}"])
        assert dt <= 1e-4 and ang <= 1e-5, (k, dt, ang)
        # the motion prior handed to the frame is the pose the reference's CV initialisation handed to it
        if k == 1:
            np.testing.assert_array_equal(b["init_rpose"], g["init_rpose_1"])
        else:
            dt, ang = pose_errors(b["init_rpose"], g[f"init_rpose_{k}"])
            assert dt <= 1e-4 and ang <= 1e-5, (k, "init_rpose", dt, ang)
    assert ours.get_relative_poses().shape == tuple(g["relative_poses_shape"]) == (FRAMES, 4, 4)
    assert len(ours.elapsed) == FRAMES and ours.get_elapsed() > 0.0
    assert ours.pointcloud_key() == "odometry_pc" and ours.relative_pose_key() == "odometry_pose"


class ObjectLoaderEnum:
    """Stand-in with the interface of the reference's loader base (slam/common/utils.py): a member's value is
    (algorithm class, config class), `load` picks the member named by the config's `type_name()` field."""

    @classmethod
    def load(cls, config, **kwargs):
        algorithm, _ = cls.__members__[getattr(config, cls.type_name())].value
        return algorithm(config, **kwargs)


def test_hydra_config_node_and_yaml(b200, golden, monkeypatch):
    _, meta = golden
    from pylidar_slam_b200 import integration
    # the shipped yaml is the reference's icp_odometry.yaml with the algorithm renamed
    ours = yaml.safe_load(open(os.path.join(integration.CONFIG_DIR, "slam", "odometry", "icp_odometry_b200.yaml")))
    theirs = dict(meta["icp_odometry_yaml"])
    assert ours.pop("algorithm") == "icp_F2M_b200" and theirs.pop("algorithm") == "icp_F2M"
    assert ours == theirs
    # the config class carries the reference's defaults, except the device the odometry runs on
    defaults = b200.ICPFrameToModelConfig()
    for name, value in meta["config_defaults"].items():
        if name != "device":
            assert getattr(defaults, name) == value, (name, getattr(defaults, name), value)

    # the hydra node: ConfigStore.store as hydra.core.config_store has it
    class ConfigStore:
        repo = {}

        @classmethod
        def instance(cls):
            return cls

        @classmethod
        def store(cls, name, node, group=None, **kwargs):
            cls.repo[f"{group}/{name}.yaml"] = node

    store = types.ModuleType("hydra.core.config_store")
    store.ConfigStore = ConfigStore
    for name in ("hydra", "hydra.core"):
        monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
    monkeypatch.setitem(sys.modules, "hydra.core.config_store", store)
    cs = integration.register_hydra_configs(b200.ICPFrameToModelConfig)
    node = cs.repo["slam/odometry/icp_odometry_b200.yaml"]
    assert node.algorithm == "icp_F2M_b200" and node.data_key == meta["config_defaults"]["data_key"]

    # the registry: the reference's ODOMETRY enum plus one member resolves the new name to this package's class
    class ODOMETRY(ObjectLoaderEnum, Enum):
        icp_F2M = (None, b200.ICPFrameToModelConfig)

        @classmethod
        def type_name(cls):
            return "algorithm"

    patched = integration.patched_odometry_enum(ODOMETRY, b200.ICPFrameToModelConfig)
    assert "icp_F2M_b200" in patched.__members__ and "icp_F2M" in patched.__members__
    algo = patched.load(b200.ICPFrameToModelConfig(algorithm="icp_F2M_b200", local_map=b200.KdTreeLocalMapConfig(),
                                                   alignment=b200.GaussNewtonPointToPlaneConfig()), **_loader_kwargs(b200))
    assert type(algo).__module__ == "pylidar_slam_b200.odometry"
    assert algo.config.local_map.type == "kdtree_local_map"
    assert algo.config.max_num_alignments == meta["config_defaults"]["max_num_alignments"] == 100


def test_reference_alignments_cannot_apply_a_mask(b200, golden):
    """Why pylidar_slam_b200's alignments answer a `mask` with a RuntimeError: the reference does (its cost functions
    multiply the [b,n,6] Jacobian in place by mask.unsqueeze(1), optimization.py:391-392,500-501)."""
    _, meta = golden
    for name in ("point_to_plane", "point_to_point"):
        err = meta["mask_errors"][name]
        assert err is not None and err["type"] == "RuntimeError" and "broadcast" in err["message"], (name, err)
    n = 128
    rs = np.random.RandomState(3)
    pts = torch.from_numpy(rs.randn(1, n, 3).astype(np.float32))
    nrm = torch.nn.functional.normalize(torch.from_numpy(rs.randn(1, n, 3).astype(np.float32)), dim=2)
    mask = torch.ones(1, n, 1)
    gn = dict(scheme="geman_mcclure", sigma=0.3, max_iters=1)
    plane = b200.GaussNewtonPointToPlaneAlignment(b200.GaussNewtonPointToPlaneConfig(gauss_newton_config=gn))
    point = b200.GaussNewtonPointToPointAlignment(b200.GNPointToPointConfig(gauss_newton_config=gn))
    with pytest.raises(RuntimeError, match="broadcast"):
        plane.align(pts, pts + 0.01, nrm, mask=mask)
    with pytest.raises(RuntimeError, match="broadcast"):
        point.align(pts, pts + 0.01, mask=mask)
