"""Pins the plain-C oracle (oracle/karto_port.c) against the reference: the unmodified karto_sdk, through the committed
golden fixtures generated from it (tests/golden/make_golden.py, tests/golden/make_reference_golden.py)."""
import hashlib
import math
import os

import numpy as np
import pytest

import helpers as H
from oracle import karto_port as P
from slam_toolbox_b200 import synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "matcher_golden.npz")
REF_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_matcher_golden.npz")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def golden_case(z, key):
    """inputs of one case of reference_matcher_golden.npz"""
    return dict(base_ranges=H.golden_ranges(z, f"{key}/base_ranges"), base_poses=z[f"{key}/base_poses"],
                query_ranges=H.golden_ranges(z, f"{key}/query_ranges"), query_pose=z[f"{key}/query_pose"])


def golden_cases():
    z = np.load(GOLDEN)
    names = sorted({k.split("/")[0] for k in z.files})
    return z, names


CONFIG = {"seq_k03": (H.MAPPER_SEQ, H.GRID_SEQ), "seq_yaml_inf": (H.MAPPER_SEQ, H.GRID_SEQ_YAML),
          "loop_chain5": (H.MAPPER_LOOP, H.GRID_LOOP), "loop_refine": (H.MAPPER_LOOP, H.GRID_LOOP),
          "small": (H.MAPPER_LOOP, H.GRID_SMALL)}


@pytest.mark.parametrize("name", sorted(CONFIG))
def test_port_matches_golden(name):
    z, _ = golden_cases()
    mapper, grid = CONFIG[name]
    pm = H.port_matcher(mapper, grid)
    base = H.port_scans(z[f"{name}/base_ranges"], z[f"{name}/base_poses"])
    q = H.port_scans(z[f"{name}/query_ranges"], z[f"{name}/query_pose"])[0]
    pen, refine = (bool(v) for v in z[f"{name}/flags"])
    resp, mean, cov = pm.match(q, base, pen, refine)
    assert resp == z[f"{name}/response"][0]
    assert np.array_equal(mean, z[f"{name}/mean"])
    assert np.array_equal(cov, z[f"{name}/cov"])
    assert np.array_equal(pm.kernel(), z[f"{name}/kernel"])
    pm.raster(q, base)
    assert sha(pm.grid()["data"]) == z[f"{name}/grid_sha"][0]
    off = pm.offsets(q, z[f"{name}/query_pose"][2], mapper["coarse_search_angle_offset"], mapper["coarse_angle_resolution"])
    assert sha(off) == z[f"{name}/offsets_sha"][0]
    so, sr = H.coarse_search(grid)
    _, _, _, vol = pm.correlate(q, z[f"{name}/query_pose"], so, sr, mapper["coarse_search_angle_offset"],
                                mapper["coarse_angle_resolution"], False, False)
    assert sha(vol) == z[f"{name}/volume_sha"][0]
    assert int(vol.argmax()) == z[f"{name}/volume_argmax"][0] and int(vol.max()) == z[f"{name}/volume_argmax"][1]


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("cfg", ["seq", "seq_yaml", "loop"])
def test_port_vs_reference_match(seed, cfg):
    z, key = np.load(REF_GOLDEN), f"match/{cfg}/{seed}"
    mapper, grid = {"seq": (H.MAPPER_SEQ, H.GRID_SEQ), "seq_yaml": (H.MAPPER_SEQ, H.GRID_SEQ_YAML),
                    "loop": (H.MAPPER_LOOP, H.GRID_LOOP)}[cfg]
    case = golden_case(z, f"case{seed}")
    pm = H.port_matcher(mapper, grid)
    pb, pq = H.port_scans(case["base_ranges"], case["base_poses"]), H.port_scans(case["query_ranges"], case["query_pose"])[0]
    assert H.digest(pq.points) == z[f"case{seed}/query_points_sha"][0]
    for i, (pen, refine) in enumerate(((True, True), (False, False), (False, True))):
        b = pm.match(pq, pb, pen, refine)
        assert z[f"{key}/response"][i] == b[0] and np.array_equal(z[f"{key}/mean"][i], b[1]) and np.array_equal(z[f"{key}/cov"][i], b[2])
    g = pm.grid()
    assert H.digest(g["data"]) == z[f"{key}/grid_sha"][0] and g["offset"] == tuple(z[f"{key}/grid_offset"])
    assert [g["width"], g["stride"], *g["roi"], g["kernel_size"]] == list(z[f"{key}/grid_geometry"])
    assert np.array_equal(z[f"{key}/kernel"], pm.kernel())
    o = pm.offsets(pq, case["query_pose"][2] + 0.01, mapper["coarse_search_angle_offset"], mapper["coarse_angle_resolution"])
    assert H.digest(o) == z[f"{key}/offsets_sha"][0]
    vp = case["query_pose"][:2] + 0.3
    assert [H.digest(P.find_valid_points(p_s, vp)) for p_s in pb] == list(z[f"{key}/valid_points_sha"])


def test_port_vs_reference_edge_cases():
    z = np.load(REF_GOLDEN)
    pm = H.port_matcher(H.MAPPER_LOOP, H.GRID_SMALL)
    case = golden_case(z, "edge")
    pq = H.port_scans(case["query_ranges"], case["query_pose"])[0]
    pb = H.port_scans(case["base_ranges"], case["base_poses"])

    def same(name, b):
        a = [z[f"edge/{name}/response"][0], z[f"edge/{name}/mean"], z[f"edge/{name}/cov"]]
        return a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    # no base scans at all: zero response everywhere, every pose ties, response expansion kicks in
    b = pm.match(pq, [], True, True)
    assert z["edge/empty/response"][0] == b[0] == 0.0 and same("empty", b)
    # all-invalid query readings
    bad = np.full_like(case["query_ranges"], np.inf)
    assert same("bad_query", pm.match(H.port_scans(bad, case["query_pose"])[0], pb, False, False))
    # query far away from the base scans (nothing overlaps)
    far = case["query_pose"] + np.array([500.0, -300.0, 1.0])
    assert same("far_query", pm.match(H.port_scans(case["query_ranges"], far)[0], pb, True, False))


def test_raster_order_dependence_is_reproduced():
    """SURVEY.md 7 hard part 2: with smear 0.1 @ 0.01 m the grid depends on base-scan order."""
    z = np.load(REF_GOLDEN)
    case = golden_case(z, "raster")
    pm = H.port_matcher(H.MAPPER_SEQ, H.GRID_SEQ_YAML)
    pq = H.port_scans(case["query_ranges"], case["query_pose"])[0]
    pb = H.port_scans(case["base_ranges"], case["base_poses"])
    grids = []
    for order, ref_sha in zip((slice(None), slice(None, None, -1)), z["raster/grid_sha"]):
        pm.raster(pq, pb[order])
        assert H.digest(pm.grid()["data"]) == ref_sha
        grids.append(pm.grid()["data"])
    assert not np.array_equal(grids[0], grids[1])


def test_create_rejects_what_the_reference_rejects():
    for bad in (dict(search_size=-1.0), dict(resolution=0.0), dict(smear_deviation=-0.1), dict(range_threshold=0.0),
                dict(smear_deviation=1.0), dict(smear_deviation=0.001)):
        kw = dict(search_size=1.0, resolution=0.05, smear_deviation=0.03, range_threshold=6.0, coarse_search_angle_offset=0.3,
                  coarse_angle_resolution=0.03, fine_search_angle_offset=0.003, distance_variance_penalty=0.25,
                  angle_variance_penalty=1.0, minimum_distance_penalty=0.5, minimum_angle_penalty=0.9, use_response_expansion=0)
        kw.update(bad)
        with pytest.raises(ValueError):
            P.PortMatcher(**kw)
