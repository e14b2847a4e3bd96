"""cfg3 (reduced): the reference's own karto::Mapper::Process replayed over a posed-scan sequence, once with the
reference CPU ScanMatcher and once with every MatchScan redirected to the GPU through the link-time seam
(integration/scan_matcher_b200.cpp), both with the GPU ScanSolver adapter installed. Because the GPU matcher is
bit-identical to the reference, the two SLAM runs must produce identical graphs and identical poses."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "integration"))
import replay  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not replay.available(), reason="integration/_build/ is built only where the reference sources are present")]


def test_mapper_process_replay_is_identical_with_the_gpu_matcher():
    ranges, odom, truth = replay.make_trajectory(4, 120)
    params = dict(replay.YAML_PARAMS, correlation_search_space_smear_deviation=0.03, loop_search_space_dimension=4.0)
    a = replay.run("ref", ranges, odom, params)
    b = replay.run("b200", ranges, odom, params, map_resolution=0.05)
    assert a["scans"] == b["scans"] and a["scans"] > 50
    assert np.array_equal(a["kept"], b["kept"])
    assert a["edges"] == b["edges"] and a["solver_computes"] == b["solver_computes"]
    assert np.array_equal(a["poses"], b["poses"])
    assert b["match_calls"] >= b["scans"] - 1
    # ScanSolver::getGraph() of the adapter (the node store the toolbox visualises): one finite pose per vertex
    assert b["graph_nodes"] == b["scans"] and len(np.unique(b["graph_ids"])) == b["scans"] and np.isfinite(b["graph_poses"]).all()
    # the published map (SMapper::getOccupancyGrid): b200og binding == the reference's OccupancyGrid::CreateFromScans
    assert b["map_cpu_seconds"] >= 0 and b["map_gpu_seconds"] >= 0
    assert np.array_equal(b["map_cpu_dims"], b["map_gpu_dims"]) and np.array_equal(b["map_cpu_offset"], b["map_gpu_offset"])
    assert np.array_equal(b["map_cpu_cells"], b["map_gpu_cells"]) and (b["map_gpu_cells"] == 100).sum() > 100
    # the matcher actually corrected the drifting odometry
    kept = a["kept"]
    err_odo = np.abs(odom[kept, :2] - truth[kept, :2]).max()
    err_slam = np.abs(a["poses"][:, :2] - truth[kept, :2] - (a["poses"][0, :2] - truth[kept[0], :2])).max()
    assert err_slam < err_odo


def test_replay_with_the_shipped_yaml_parameters_order_dependent_raster():
    """smear 0.1 m @ 0.01 m (config/mapper_params_online_sync.yaml): the raster depends on insertion order."""
    ranges, odom, _ = replay.make_trajectory(5, 40)
    a = replay.run("ref", ranges, odom, replay.YAML_PARAMS)
    b = replay.run("b200", ranges, odom, replay.YAML_PARAMS)
    assert a["scans"] == b["scans"] and np.array_equal(a["poses"], b["poses"]) and a["edges"] == b["edges"]


def test_adapter_option_mapping_and_handle_lifetime():
    """B200Solver::ConfigureFromStrings maps the ceres_* keys of CeresSolver::Configure (solvers/ceres_solver.cpp:25-193); the matcher
    shim's ~ScanMatcher releases the device state when Mapper::Reset / ~Mapper delete the matchers (no leak, no stale aliases)."""
    import json
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "integration", "replay.py"), "lifecycle"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    c = out["configure"]
    assert c["ceres_loss_function=HuberLoss"] == 1 and c["ceres_loss_function=CauchyLoss"] == 1 and c["ceres_loss_function=None"] == 1
    assert c["ceres_loss_function=Bogus"] == 0 and c["ceres_trust_strategy=DOGLEG"] == 0 and c["no_such_key=1"] == 0
    assert c["ceres_trust_strategy=LEVENBERG_MARQUARDT"] == 1 and c["ceres_linear_solver=SPARSE_NORMAL_CHOLESKY"] == 1
    assert out["live_handles"] == [0, 2, 0, 2, 0], out["live_handles"]
