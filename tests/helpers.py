"""Shared fixtures for the parity tests: the parameter sets of BASELINE.json's configs and
constructors for the three implementations (reference .so, C port oracle, CUDA product), and the codec of the laser
ranges stored in the golden fixtures."""
from __future__ import annotations

import math

import numpy as np

from slam_toolbox_b200 import synth

LASER = dict(min_angle=synth.ANGLE_MIN, max_angle=synth.ANGLE_MAX, ang_res=synth.ANGLE_INC, min_range=0.1, max_range=30.0,
             range_threshold=12.0)

# toolbox-style parameter values (before the setters square the variance penalties)
MAPPER_SEQ = dict(coarse_search_angle_offset=math.radians(5.0), coarse_angle_resolution=math.radians(2.0),
                  fine_search_angle_offset=math.radians(0.2), distance_variance_penalty=0.5, angle_variance_penalty=1.0,
                  minimum_distance_penalty=0.5, minimum_angle_penalty=0.9, use_response_expansion=1)
MAPPER_LOOP = dict(MAPPER_SEQ, coarse_search_angle_offset=math.radians(20.0))

# ScanMatcher::Create arguments: (searchSize, resolution, smearDeviation, rangeThreshold)
GRID_SEQ = (1.0, 0.01, 0.03, 12.0)       # cfg1, Karto smear
GRID_SEQ_YAML = (1.0, 0.01, 0.1, 12.0)   # cfg1, shipped YAML smear (order-dependent raster)
GRID_LOOP = (4.0, 0.05, 0.03, 12.0)      # cfg2 / cfg5
GRID_SMALL = (0.5, 0.05, 0.03, 6.0)      # small fast case for unit tests


def ref_matcher(mapper_kw, grid):
    from oracle import karto_ref as R
    R.init_laser(**LASER)
    return R.RefMatcher(R.RefMapper(**mapper_kw), *grid)


def port_matcher(mapper_kw, grid):
    from oracle import karto_port as P
    return P.PortMatcher(search_size=grid[0], resolution=grid[1], smear_deviation=grid[2], range_threshold=grid[3],
                         coarse_search_angle_offset=mapper_kw["coarse_search_angle_offset"],
                         coarse_angle_resolution=mapper_kw["coarse_angle_resolution"],
                         fine_search_angle_offset=mapper_kw["fine_search_angle_offset"],
                         distance_variance_penalty=mapper_kw["distance_variance_penalty"] ** 2,
                         angle_variance_penalty=mapper_kw["angle_variance_penalty"] ** 2,
                         minimum_distance_penalty=mapper_kw["minimum_distance_penalty"],
                         minimum_angle_penalty=mapper_kw["minimum_angle_penalty"],
                         use_response_expansion=int(mapper_kw["use_response_expansion"]))


def gpu_matcher(mapper_kw, grid):
    from slam_toolbox_b200 import api
    mp = api.MapperParams(**{k: (bool(v) if k == "use_response_expansion" else v) for k, v in mapper_kw.items()})
    return api.ScanMatcher.Create(mp, *grid)


def port_scans(ranges, poses):
    from oracle import karto_port as P
    return [P.PortScan(r, p, synth.ANGLE_MIN, synth.ANGLE_INC) for r, p in zip(np.atleast_2d(ranges), np.atleast_2d(poses))]


def ref_scans(ranges, poses, uid0=0):
    from oracle import karto_ref as R
    R.init_laser(**LASER)
    return [R.RefScan(r, p, uid0 + i) for i, (r, p) in enumerate(zip(np.atleast_2d(ranges), np.atleast_2d(poses)))]


def coarse_search(grid):
    """(searchSpaceOffset, searchSpaceResolution) of MatchScan's coarse pass (Mapper.cpp:577-585)."""
    side = math.floor(grid[0] / grid[1] + 0.5) + 1
    res = 1.0 / (1.0 / grid[1])
    off = 0.5 * (side - 1) * res
    return (off, off), (2 * res, 2 * res)


def gpu_block(ranges, poses, range_threshold=None):
    from slam_toolbox_b200 import api
    laser = api.LaserRangeFinder(minimum_angle=LASER["min_angle"], maximum_angle=LASER["max_angle"], angular_resolution=LASER["ang_res"],
                                 minimum_range=LASER["min_range"], maximum_range=LASER["max_range"],
                                 range_threshold=LASER["range_threshold"] if range_threshold is None else range_threshold)
    return api.ScanBlock(ranges, poses, laser)


def digest(a) -> str:
    """SHA-256 of an array's bytes, NaNs canonicalised first: equal digests mean np.array_equal(..., equal_nan=True)."""
    import hashlib
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a)
    return hashlib.sha256(a.tobytes()).hexdigest()


# laser ranges in the golden fixtures: uint16 millimetres, three codes reserved for +inf, NaN and readings that are not a
# whole number of millimetres (their exact float64 values are stored separately, in order)
RANGE_INF, RANGE_NAN, RANGE_EXACT = 65535, 65534, 65533


def pack_ranges(r):
    r = np.asarray(r, dtype=np.float64)
    finite = np.isfinite(r)
    assert not (np.isinf(r) & (r < 0)).any() and (r[finite] >= 0).all() and (r[finite] < RANGE_EXACT / 1000.0).all()
    mm = np.round(np.where(finite, r, 0.0) * 1000.0)
    exact = finite & (mm / 1000.0 != r)
    codes = np.where(np.isnan(r), RANGE_NAN, np.where(np.isinf(r), RANGE_INF, np.where(exact, RANGE_EXACT, mm)))
    return codes.astype(np.uint16), r[exact]


def unpack_ranges(codes, exact):
    r = codes.astype(np.float64) / 1000.0
    r[codes == RANGE_INF] = np.inf
    r[codes == RANGE_NAN] = np.nan
    r[codes == RANGE_EXACT] = exact
    return r


def golden_ranges(z, key):
    """The ranges stored under `key` by pack_ranges (keys <key>_mm and <key>_exact)."""
    return unpack_ranges(z[f"{key}_mm"], z[f"{key}_exact"])


def assert_occupancy_equals_golden(g, z, name):
    """g = dict(width, height, stride, offset, cells, passes, hits) vs tests/golden/occupancy_golden.npz case `name`"""
    import hashlib
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()   # noqa: E731
    assert [g["width"], g["height"], g["stride"]] == list(z[f"{name}/dims"])
    assert np.array_equal(g["offset"], z[f"{name}/offset"])
    assert np.array_equal(g["cells"], z[f"{name}/cells"])
    assert [int(g["passes"].sum()), int(g["hits"].sum())] == list(z[f"{name}/sums"])
    assert sha(g["passes"].astype(np.uint32)) == z[f"{name}/pass_sha"][0]
    assert sha(g["hits"].astype(np.uint32)) == z[f"{name}/hits_sha"][0]
