"""Occupancy grid (karto::OccupancyGrid::CreateFromScans, Karto.h:5946-5961): pins the plain-C oracle
(kp_occupancy_create) against the committed fixtures generated from the unmodified reference
(tests/golden/make_occupancy_golden.py, tests/golden/make_reference_golden.py)."""
import hashlib
import os

import numpy as np
import pytest

import helpers as H
from oracle import karto_port as P
from slam_toolbox_b200 import synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "occupancy_golden.npz")
REF_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_occupancy_golden.npz")
CASES = ["coarse_strict", "default", "one_scan", "short_threshold"]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def port_grid(ranges, poses, res, rt, mp, th):
    return P.occupancy(H.port_scans(ranges, poses), res, rt, H.LASER["min_range"], H.LASER["max_range"],
                       2 if mp < 0 else int(mp), 0.1 if th < 0 else th)


@pytest.mark.parametrize("name", CASES)
def test_port_matches_golden(name):
    z = np.load(GOLDEN)
    res, rt, mp, th = z[f"{name}/params"]
    g = port_grid(z[f"{name}/ranges"], z[f"{name}/poses"], res, rt, mp, th)
    H.assert_occupancy_equals_golden(g, z, name)


@pytest.mark.parametrize("seed,n,res,mp,th", [(0, 30, 0.05, -1, -1.0), (1, 20, 0.1, 4, 0.25), (2, 12, 0.02, 0, 0.05)])
def test_port_vs_reference(seed, n, res, mp, th):
    z, key = np.load(REF_GOLDEN), f"run{seed}"
    ranges, poses = H.golden_ranges(z, f"{key}/ranges"), z[f"{key}/poses"]
    assert len(ranges) == len(poses) == n
    b = port_grid(ranges, poses, res, H.LASER["range_threshold"], mp, th)
    assert [b["width"], b["height"], b["stride"]] == list(z[f"{key}/dims"])
    assert np.array_equal(b["offset"], z[f"{key}/offset"])
    assert H.digest(b["cells"]) == z[f"{key}/cells_sha"][0]
    assert H.digest(b["passes"]) == z[f"{key}/pass_sha"][0] and H.digest(b["hits"]) == z[f"{key}/hits_sha"][0]
    occupied, free, passes, hits = z[f"{key}/counts"]
    assert [(b["cells"] == 100).sum(), (b["cells"] == 255).sum(), b["passes"].sum(), b["hits"].sum()] == [occupied, free, passes, hits]
    assert occupied > 50 and free > 1000


def test_no_scans_is_null():
    assert np.load(REF_GOLDEN)["no_scans/is_null"][0]          # Karto.h:5950-5952
    assert P.occupancy([], 0.05, 12.0, 0.1, 30.0) is None


def test_counters_are_consistent():
    """every hit is also a pass; cells follow UpdateCell (Karto.h:6241-6254) from the counters"""
    run = synth.make_mapping_run(7, 10)
    g = port_grid(run["ranges"], run["poses"], 0.05, 12.0, 2, 0.1)
    ps, ht = g["passes"].astype(np.int64), g["hits"].astype(np.int64)
    assert (ht <= ps).all()
    exp = np.zeros_like(g["cells"])
    known = ps > 2
    ratio = np.divide(ht, ps, out=np.zeros(ps.shape), where=ps > 0)
    exp[known & (ratio > 0.1)] = 100
    exp[known & ~(ratio > 0.1)] = 255
    assert np.array_equal(exp, g["cells"])
    assert not g["cells"][:, g["width"]:].any()   # width-step padding is never touched
