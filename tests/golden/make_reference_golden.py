"""Generates the reference_*_golden.npz fixtures from the UNMODIFIED reference (oracle/_ref/libkarto_ref.so, built by
oracle/Makefile where the reference sources are present):
    python tests/golden/make_reference_golden.py
They record what the reference returned for the inputs of the port-vs-reference tests, so that those tests pin the
C-port oracle against the reference on any machine, with or without the reference library:

  reference_matcher_golden.npz    test_oracle_vs_ref.py: MatchScan results, correlation-grid / lookup-table / valid-point
                                  digests, the order-dependent raster, the edge cases
  reference_occupancy_golden.npz  test_occupancy_oracle.py: OccupancyGrid::CreateFromScans cells and counters, NULL on no scans
  reference_posegraph_golden.npz  test_posegraph_oracle.py: LinkInfo and Matrix3::Inverse

Every case stores its inputs next to the reference's outputs.  The synthetic ranges are rounded to whole millimetres
before the reference sees them (helpers.pack_ranges stores them in two bytes each); the readings make_mapping_run
places on purpose just inside the range threshold keep their exact value.  Large outputs are stored as digests
(helpers.digest)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import helpers as H  # noqa: E402
from helpers import digest  # noqa: E402
from oracle import karto_ref as R  # noqa: E402
from slam_toolbox_b200 import synth  # noqa: E402

MATCH_CFGS = {"seq": (H.MAPPER_SEQ, H.GRID_SEQ), "seq_yaml": (H.MAPPER_SEQ, H.GRID_SEQ_YAML), "loop": (H.MAPPER_LOOP, H.GRID_LOOP)}
MATCH_SEEDS = (0, 1, 2)
MATCH_FLAGS = ((True, True), (False, False), (False, True))       # (penalize, refine), in the order the test matches
OCC_CASES = [(0, 30, 0.05, -1, -1.0), (1, 20, 0.1, 4, 0.25), (2, 12, 0.02, 0, 0.05)]   # seed, scans, res, min_pass, threshold
KEEP_EXACT = (12.0 - 5e-7,)      # make_mapping_run's reading inside the KT_TOLERANCE band of the range threshold


def millimetres(r):
    r = np.asarray(r, dtype=np.float64)
    q = np.round(np.where(np.isfinite(r), r, 0.0) * 1000.0) / 1000.0
    return np.where(np.isfinite(r) & ~np.isin(r, KEEP_EXACT), q, r)


def put_ranges(out, key, r):
    out[f"{key}_mm"], out[f"{key}_exact"] = H.pack_ranges(r)
    assert np.array_equal(H.golden_ranges(out, key), r, equal_nan=True)


def sequential_case(out, key, seed, **kw):
    case = synth.make_sequential_case(seed, **kw)
    case["base_ranges"], case["query_ranges"] = millimetres(case["base_ranges"]), millimetres(case["query_ranges"])
    put_ranges(out, f"{key}/base_ranges", case["base_ranges"])
    put_ranges(out, f"{key}/query_ranges", case["query_ranges"])
    out[f"{key}/base_poses"], out[f"{key}/query_pose"] = case["base_poses"], case["query_pose"]
    return case


def matcher():
    out = {}
    for seed in MATCH_SEEDS:
        case = sequential_case(out, f"case{seed}", 100 + seed, buffer_len=4, inf_frac=0.03 * (seed % 2), nan_frac=0.01 * (seed == 2))
        rq = H.ref_scans(case["query_ranges"], case["query_pose"], 99)[0]
        out[f"case{seed}/query_points_sha"] = np.array([digest(rq.points())])
        for cfg, (mapper, grid) in MATCH_CFGS.items():
            key = f"match/{cfg}/{seed}"
            rm = H.ref_matcher(mapper, grid)
            rb = H.ref_scans(case["base_ranges"], case["base_poses"])
            rq = H.ref_scans(case["query_ranges"], case["query_pose"], 99)[0]
            res = [rm.match(rq, rb, pen, refine) for pen, refine in MATCH_FLAGS]
            out[f"{key}/response"] = np.array([r[0] for r in res])
            out[f"{key}/mean"] = np.stack([r[1] for r in res])
            out[f"{key}/cov"] = np.stack([r[2] for r in res])
            g = rm.grid()
            out[f"{key}/grid_sha"] = np.array([digest(g["data"])])
            out[f"{key}/grid_offset"] = np.array(g["offset"])
            out[f"{key}/grid_geometry"] = np.array([g["width"], g["stride"], *g["roi"], g["kernel_size"]])
            out[f"{key}/kernel"] = rm.kernel()
            off = rm.offsets(rq, case["query_pose"][2] + 0.01, mapper["coarse_search_angle_offset"], mapper["coarse_angle_resolution"])
            out[f"{key}/offsets_sha"] = np.array([digest(off)])
            vp = case["query_pose"][:2] + 0.3
            out[f"{key}/valid_points_sha"] = np.array([digest(rm.find_valid_points(s, vp)) for s in rb])
            print(key, "responses", out[f"{key}/response"])

    # edge cases: no base scans, an all-invalid query, a query far away from every base scan
    rm = H.ref_matcher(H.MAPPER_LOOP, H.GRID_SMALL)
    case = sequential_case(out, "edge", 7, buffer_len=2)
    rq = H.ref_scans(case["query_ranges"], case["query_pose"], 5)[0]
    rb = H.ref_scans(case["base_ranges"], case["base_poses"])
    bad = np.full_like(case["query_ranges"], np.inf)
    far = case["query_pose"] + np.array([500.0, -300.0, 1.0])
    for name, q, base, pen, refine in (("empty", rq, [], True, True),
                                       ("bad_query", H.ref_scans(bad, case["query_pose"], 6)[0], rb, False, False),
                                       ("far_query", H.ref_scans(case["query_ranges"], far, 7)[0], rb, True, False)):
        r, m, c = rm.match(q, base, pen, refine)
        out[f"edge/{name}/response"], out[f"edge/{name}/mean"], out[f"edge/{name}/cov"] = np.array([r]), m, c
        print("edge", name, r)

    # smear 0.1 m @ 0.01 m: the raster depends on the order of the base scans
    case = sequential_case(out, "raster", 3, buffer_len=4)
    rm = H.ref_matcher(H.MAPPER_SEQ, H.GRID_SEQ_YAML)
    rq = H.ref_scans(case["query_ranges"], case["query_pose"], 9)[0]
    rb = H.ref_scans(case["base_ranges"], case["base_poses"])
    shas = []
    for order in (slice(None), slice(None, None, -1)):
        rm.raster(rq, rb[order])
        shas.append(digest(rm.grid()["data"]))
    out["raster/grid_sha"] = np.array(shas)
    assert shas[0] != shas[1]
    return out


def occupancy():
    out = {}
    for seed, n, res, mp, th in OCC_CASES:
        key = f"run{seed}"
        run = synth.make_mapping_run(seed, n, inf_frac=0.03)
        ranges = millimetres(run["ranges"])
        g = R.occupancy(H.ref_scans(ranges, run["poses"]), res, mp, th)
        put_ranges(out, f"{key}/ranges", ranges)
        out[f"{key}/poses"] = run["poses"]
        out[f"{key}/dims"] = np.array([g["width"], g["height"], g["stride"]])
        out[f"{key}/offset"] = g["offset"]
        out[f"{key}/cells_sha"] = np.array([digest(g["cells"])])
        out[f"{key}/pass_sha"] = np.array([digest(g["passes"])])
        out[f"{key}/hits_sha"] = np.array([digest(g["hits"])])
        out[f"{key}/counts"] = np.array([int((g["cells"] == 100).sum()), int((g["cells"] == 255).sum()),
                                         int(g["passes"].sum()), int(g["hits"].sum())])
        print(key, (g["width"], g["height"], g["stride"]), "occupied, free, passes, hits", out[f"{key}/counts"])
    R.init_laser(**H.LASER)
    out["no_scans/is_null"] = np.array([R.occupancy([], 0.05) is None])
    return out


def posegraph():
    rng = np.random.default_rng(0)
    p1s, p2s, covs, ds, cs, invs = [], [], [], [], [], []
    for _ in range(20):
        p1, p2 = rng.uniform(-5, 5, 3), rng.uniform(-5, 5, 3)
        A = rng.normal(size=(3, 3))
        cov = A @ A.T + 0.1 * np.eye(3)
        d, c = R.link_info(p1, p2, cov)
        p1s.append(p1); p2s.append(p2); covs.append(cov); ds.append(d); cs.append(c); invs.append(R.matrix3_inverse(cov))
    return {"p1": np.stack(p1s), "p2": np.stack(p2s), "cov": np.stack(covs), "link_delta": np.stack(ds), "link_cov": np.stack(cs),
            "inverse": np.stack(invs)}


def main():
    assert R.available(), "oracle/_ref/libkarto_ref.so is not built"
    for name, make in (("matcher", matcher), ("occupancy", occupancy), ("posegraph", posegraph)):
        path = os.path.join(HERE, f"reference_{name}_golden.npz")
        np.savez_compressed(path, **make())
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
