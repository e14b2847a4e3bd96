#!/usr/bin/env python
"""bench.py -- the hot-path benchmark of b200slam.

Metric (BASELINE.json): scan matches/sec (1081-beam, +-2 m / +-20 deg) on the loop-closure
batch workload (configs[1]: 1 query x 1000 candidate 1081-beam scans per GPU), plus the
10k-node / 40k-edge SE(2) pose-graph solve time (configs[3]) reported in the same JSON line
under "graph_solve", and the map-publish step (occupancy grid from 5,000 scans) under "occupancy_grid".

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path
                                                           # (oracle/_ref = unmodified karto_sdk)
  python bench.py ... --dump-outputs DIR                   # also write what the timed path computed in its
                                                           # last step as DIR/<name>.npy (see dump_outputs)

One "step" = one pass of the hot path over one batch: every rank sweeps its shard of candidate
chains (rasterise + exhaustive (x, y, theta) correlation + reduction for each (query, chain)
pair) and, for N > 1, joins the per-query best-response all-reduce (NCCL, MAX of a packed key).
  value  : pairs matched by all ranks / device time, inputs already resident in HBM
  e2e    : the same through the public API call (ScanMatcher.MatchScanBatch) with HOST inputs
           (pinned), host<->device copies inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scan matches/sec (1081-beam, +-2m/+-20deg)"
UNIT = "matches/s"

# cfg2 / cfg5 parameters (SURVEY.md 8d): loop matcher, search 4.0 m @ 0.05 m, smear 0.03, +-20 deg / 2 deg
LOOP_GRID = (4.0, 0.05, 0.03, 12.0)
LOOP_MAPPER = dict(coarse_search_angle_offset=math.radians(20.0), coarse_angle_resolution=math.radians(2.0),
                   fine_search_angle_offset=math.radians(0.2), distance_variance_penalty=0.5, angle_variance_penalty=1.0,
                   minimum_distance_penalty=0.5, minimum_angle_penalty=0.9, use_response_expansion=0)
N_CAND = 1000       # candidate chains per GPU per step
CHAIN_LEN = 1
N_QUERY = 1
GRAPH_NODES, GRAPH_EDGES = 10000, 40000
GRAPH_SIGMA = (0.03, 0.01)


def algorithmic_bytes_per_match(n_beams: int, n_angles: int, npairs: int, nq: int) -> float:
    """SURVEY.md 8(d): compulsory bytes of one LOOP coarse match = the 320,920 B correlation grid it
    is matched against + 128 B of outputs + the query's lookup table (n_angles x n_beams int32)
    amortised over the pairs that share it."""
    grid_bytes = 568 * 565
    return grid_bytes + 128 + (n_angles * n_beams * 4) * nq / max(npairs, 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first(self, timeout: float = 5.0):
        t = time.time()
        while self.proc and not self.lines and time.time() - t < timeout:
            time.sleep(0.02)
        self.mark = len(self.lines)   # samples from here on fall inside the timed region

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines[max(0, getattr(self, "mark", 0) - 1):]
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict) -> None:
    """--dump-outputs: writes each array as <directory>/<name>.npy.  Every input of the benchmark comes from fixed seeds,
    so two builds run with the same arguments can be compared output for output.  Float64 values and integer counters
    are written as float64 (exact), 8-bit cells as float32."""
    out = {name: np.asarray(a, dtype=np.float32 if np.asarray(a).dtype == np.uint8 else np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_LIMIT_BYTES}")
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def make_inputs(rank: int, n_cand: int, chain_len: int, n_query: int):
    from slam_toolbox_b200 import synth
    # same world + queries on every rank, candidates differ per rank (sharded candidate set)
    world = synth.make_world(7)
    rng = np.random.default_rng(1234)
    qtrue = np.array([synth.free_pose(world, rng) for _ in range(n_query)])
    qranges = synth.noisy(synth.raycast(world, qtrue), rng)
    qpose = qtrue + np.column_stack([rng.normal(0, 0.5, (n_query, 2)), rng.normal(0, 0.08, n_query)])
    crng = np.random.default_rng(99 + rank)
    starts = synth.poses_near(world, qtrue[0, :2], 3.0, n_cand, crng)
    cposes = starts if chain_len == 1 else np.concatenate([synth.chain_poses(world, s, chain_len, crng) for s in starts])
    cranges = synth.noisy(synth.raycast(world, cposes), crng)
    chain_start = np.arange(0, n_cand * chain_len + 1, chain_len, dtype=np.int32)
    return qranges, qpose, cranges, cposes, chain_start


def cpu_sweep(qranges, qpose, cranges, cposes, chain_start, n_sample: int, threads: int):
    """The reference's own MatchScan (oracle/_ref, unmodified karto_sdk) over the first n_sample chains,
    one reference ScanMatcher per host thread. Returns (matches/s, kind, seconds, responses)."""
    from oracle import karto_ref as R
    from oracle import karto_port as P
    from slam_toolbox_b200 import synth
    n_sample = min(n_sample, len(chain_start) - 1)
    cs = chain_start[:n_sample + 1]
    if R.available():
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(1)
        os.dup2(devnull, 1)   # the reference prints "Registering sensor" to stdout
        try:
            R.init_laser(synth.ANGLE_MIN, synth.ANGLE_MAX, synth.ANGLE_INC, 0.1, 30.0, LOOP_GRID[3])
        finally:
            os.dup2(saved, 1); os.close(devnull); os.close(saved)
        mp = R.RefMapper(**LOOP_MAPPER)
        matchers = [R.RefMatcher(mp, *LOOP_GRID) for _ in range(threads)]
        q = R.RefScan(qranges[0], qpose[0], 100000)
        scans = [R.RefScan(cranges[i], cposes[i], i) for i in range(cs[-1])]
        global _BEST_THREADS
        if _BEST_THREADS is None:
            # the reference allocates ~1.1 MB per match and takes a shared_mutex per scan read, so it does
            # not scale to every hardware thread: give it the thread count it is fastest with
            best = (0.0, threads)
            for t in sorted({threads, max(1, threads // 2), max(1, threads // 4), min(threads, 32), min(threads, 16), min(threads, 8)}):
                k = min(n_sample, 2 * t)
                sec, _, _, _ = R.sweep(matchers[:t], q, scans, cs[:k + 1], False, False)
                if k / sec > best[0]:
                    best = (k / sec, t)
            _BEST_THREADS = best[1]
        use = min(threads, _BEST_THREADS)
        sec, resp, _, _ = R.sweep(matchers[:use], q, scans, cs, False, False)
        return n_sample / sec, "reference", sec, resp, use
    # port fallback (single thread): the plain-C restatement
    pm = P.PortMatcher(search_size=LOOP_GRID[0], resolution=LOOP_GRID[1], smear_deviation=LOOP_GRID[2], range_threshold=LOOP_GRID[3],
                       coarse_search_angle_offset=LOOP_MAPPER["coarse_search_angle_offset"],
                       coarse_angle_resolution=LOOP_MAPPER["coarse_angle_resolution"],
                       fine_search_angle_offset=LOOP_MAPPER["fine_search_angle_offset"], distance_variance_penalty=0.25,
                       angle_variance_penalty=1.0, minimum_distance_penalty=0.5, minimum_angle_penalty=0.9, use_response_expansion=0)
    q = P.PortScan(qranges[0], qpose[0], synth.ANGLE_MIN, synth.ANGLE_INC)
    scans = [P.PortScan(cranges[i], cposes[i], synth.ANGLE_MIN, synth.ANGLE_INC) for i in range(cs[-1])]
    t = time.perf_counter()
    resp = [pm.match(q, scans[cs[j]:cs[j + 1]], False, False)[0] for j in range(n_sample)]
    sec = time.perf_counter() - t
    return n_sample / sec, "port", sec, np.array(resp), 1


_BEST_THREADS = None


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    if rank != 0:
        return
    threads = host_threads()
    qr, qp, cr, cp, cs = make_inputs(0, N_CAND, CHAIN_LEN, N_QUERY)
    # every step matches all N_CAND candidates (the same config as the b200 arm: ~2 s per step on 32 threads)
    n_sample = N_CAND
    rates = []
    for i in range(args.warmup + args.steps):
        rate, kind, sec, resp, used = cpu_sweep(qr, qp, cr, cp, cs, n_sample, threads)
        if i >= args.warmup:
            rates.append((rate, sec))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"response": resp})
    value = float(np.mean([r for r, _ in rates]))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean([s for _, s in rates])), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"cfg2 loop-closure batch: {N_QUERY} query x {N_CAND} candidate 1081-beam scans, +-2m/+-20deg "
                               f"(all {n_sample} candidates per step)",
                   "search": "41x41x21 poses", "grid": "565x568 u8", "threads": used, "host_threads_available": threads},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind,
                         "sample": f"{n_sample} of {N_CAND} candidate matches per step, one ScanMatcher per host thread"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _port_matcher(grid, mapper_kw):
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


def grid_geometry(grid):
    """(width step, height) of the correlation grid ScanMatcher::Create builds (Mapper.cpp:477-522, Karto.h:4640)."""
    side = math.floor(grid[0] / grid[1] + 0.5) + 1
    margin = math.ceil(grid[3] / grid[1])
    border = int(math.floor(2.0 * grid[2] / grid[1] + 0.5)) + 1
    w = side + 2 * margin + 2 * border
    return (w + 7) // 8 * 8, w, side


def sweep_row(name, grid, n_cand, chain_len, steps, peak, stream, flush, options=None, far_fraction=0.0, n_query=1,
              parity_samples=3, cand_radius=3.0):
    """One extra workload of the batched sweep on this GPU: device-timed steps (inputs resident, L2 flushed between steps), the
    end-to-end call with host inputs, the kernel / plan that ran, the HBM roofline on SURVEY 8(d)'s algorithmic bytes for THIS
    geometry, and an exact comparison of a few pairs with the oracle."""
    import torch
    from slam_toolbox_b200 import api, synth
    world = synth.make_world(7)
    rng = np.random.default_rng(4321)
    qtrue = synth.poses_near(world, synth.free_pose(world, rng)[:2], 1.5, n_query, rng) if n_query > 1 else np.array([synth.free_pose(world, rng)])
    qr = synth.noisy(synth.raycast(world, qtrue), rng)
    qp = qtrue + np.column_stack([rng.normal(0, 0.5, (n_query, 2)), rng.normal(0, 0.08, n_query)])
    starts = synth.poses_near(world, qtrue[0, :2], cand_radius, n_cand, rng)
    cp = starts if chain_len == 1 else np.concatenate([synth.chain_poses(world, st, chain_len, rng) for st in starts])
    cr = synth.noisy(synth.raycast(world, cp, chunk=64), rng)
    if far_fraction > 0:
        far = rng.random(n_cand) < far_fraction          # candidates that do not overlap the query's search window at all
        cp = cp.copy()
        cp[np.repeat(far, chain_len), :2] += 400.0
    cs = np.arange(0, n_cand * chain_len + 1, chain_len, dtype=np.int32)
    laser = api.LaserRangeFinder()
    mapper = api.MapperParams(**{k: (bool(v) if k == "use_response_expansion" else v) for k, v in LOOP_MAPPER.items()})
    sm = api.ScanMatcher.Create(mapper, *grid)
    sm.set_stream(stream.cuda_stream)
    for k, v in (options or {}).items():
        sm.set_option(k, v)
    pts = torch.empty((cr.shape[0], cr.shape[1], 2), dtype=torch.float64).pin_memory()
    pts.numpy()[...] = api.point_readings(cr, cp, laser)
    cands, queries = api.ScanBlock(cr, cp, laser, points=pts.numpy()), api.ScanBlock(qr, qp, laser)
    npairs = sm.batch_upload(queries, cands, cs, None, False)
    info, plan = sm.batch_info(), sm.batch_tile_info()
    for _ in range(3):
        sm.batch_run()
    torch.cuda.synchronize()
    ev, kms = [], []
    for k in range(steps):
        flush.fill_(k & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); sm.batch_run(); b.record(stream)
        ev.append((a, b))
    torch.cuda.synchronize()
    step_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    kern_ms = float(sm.batch_kernel_ms())
    resp, mean, cov = sm.batch_fetch()
    stats = sm.batch_fetch_stats()
    sm.transfer_bytes(reset=True)
    sm.MatchScanBatch(queries, cands, cs, None, False, False)
    sm.transfer_bytes(reset=True)
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(max(2, steps // 2)):
        r2 = sm.MatchScanBatch(queries, cands, cs, None, False, False)
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t) / max(2, steps // 2)
    h2d, d2h = sm.transfer_bytes()
    stride, width, side = grid_geometry(grid)
    n_angles = int(math.floor(2 * LOOP_MAPPER["coarse_search_angle_offset"] / LOOP_MAPPER["coarse_angle_resolution"] + 0.5)) + 1
    nposes = (side // 2 + 1)
    bytes_match = stride * width + 128 + (n_angles * cr.shape[1] * 4) * n_query / npairs
    achieved = bytes_match * npairs / (kern_ms * 1e-3) / 1e9
    lookups = npairs * nposes * nposes * n_angles * cr.shape[1]
    ok = True
    if parity_samples:
        pm = _port_matcher(grid, LOOP_MAPPER)
        from oracle import karto_port as P
        pq = [P.PortScan(qr[i], qp[i], synth.ANGLE_MIN, synth.ANGLE_INC) for i in range(n_query)]
        picks = sorted({0, npairs - 1, int(np.argmax(resp))} | set(rng.integers(0, npairs, max(0, parity_samples - 3)).tolist()))
        for j in picks:
            q, c = divmod(j, n_cand)
            base = [P.PortScan(cr[i], cp[i], synth.ANGLE_MIN, synth.ANGLE_INC) for i in range(cs[c], cs[c + 1])]
            e = pm.match(pq[q], base, False, False)
            ok = ok and e[0] == resp[j] and np.array_equal(e[1], mean[j]) and np.array_equal(e[2], cov[j])
    sm.close()
    return {"workload": name, "grid": f"{width}x{width} u8 (stride {stride})", "search": f"{nposes}x{nposes}x{n_angles} poses",
            "pairs": int(npairs), "chain_length": chain_len, "kernel": info["kernel"],
            "plan": {k: plan[k] for k in ("cluster", "chunks", "bands", "clusters", "smem_kb")} if info["kernel"] == "tile" else None,
            "value": npairs / (step_ms * 1e-3), "unit": UNIT, "ms_per_step": step_ms, "kernel_ms": kern_ms,
            "e2e": {"value": npairs / (e2e_ms * 1e-3), "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h2d // max(2, steps // 2)),
                    "d2h_bytes_per_step": int(d2h // max(2, steps // 2))},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "algorithmic_bytes_per_match": bytes_match, "lookups_per_s": lookups / (kern_ms * 1e-3),
                         "onchip_frac_of_128B_per_clk_per_SM": lookups / (kern_ms * 1e-3) / (128 * 148 * 1.965e9)},
            "edge_beams": info["edge_beams"], "zero_volume_pairs": stats["zero_pairs"], "single_match_fallbacks": stats["fallback_pairs"],
            "best_response": float(resp.max()), "parity_exact": bool(ok and np.array_equal(r2[0], resp)),
            "parity_checked_pairs": int(len(picks)) if parity_samples else 0}


def seq_match_bench(n_matches: int, with_cpu: bool):
    """cfg1: the per-scan sequential match (Mapper.cpp:2714 -> MatchScan, coarse + fine, penalised) against a running buffer of 10
    scans, search 1.0 m @ 0.01 m, +-5 deg -- once with Karto's smear (0.03) and once with the shipped YAML's (0.1: order-dependent
    raster).  GPU: host buffers in, result out through b200sm_match (every call synchronises).  CPU: the reference's MatchScan on one
    core (its TBB row loop is a serial shim in the oracle build)."""
    from slam_toolbox_b200 import api, synth
    seq_mapper = dict(LOOP_MAPPER, coarse_search_angle_offset=math.radians(5.0), use_response_expansion=1)
    out = {}
    for tag, smear in (("smear_0.03", 0.03), ("smear_0.1_yaml", 0.1)):
        grid = (1.0, 0.01, smear, 12.0)
        laser = api.LaserRangeFinder()
        mapper = api.MapperParams(**{k: (bool(v) if k == "use_response_expansion" else v) for k, v in seq_mapper.items()})
        sm = api.ScanMatcher.Create(mapper, *grid)
        cases = [synth.make_sequential_case(100 + i, buffer_len=10) for i in range(4)]
        blocks = [(api.ScanBlock(c["query_ranges"][None, :], c["query_pose"][None, :], laser), api.ScanBlock(c["base_ranges"], c["base_poses"], laser))
                  for c in cases]
        for q, b in blocks:
            sm.MatchScan(q, b, True, True)
        l0 = sm.launch_count()
        sm.match_timing(reset=True)
        t = time.perf_counter()
        res = []
        for i in range(n_matches):
            q, b = blocks[i % len(blocks)]
            res.append(sm.MatchScan(q, b, True, True))
        gpu_ms = 1e3 * (time.perf_counter() - t) / n_matches
        row = {"grid": "%dx%d u8" % (grid_geometry(grid)[1], grid_geometry(grid)[1]), "search": "51x51x6 coarse + 3x3x11 fine",
               "gpu_ms_per_match_e2e": gpu_ms, "gpu_matches_per_s": 1e3 / gpu_ms, "launches_per_match": (sm.launch_count() - l0) / n_matches,
               "host_phases_ms": {k: round(float(v), 4) for k, v in sm.match_timing().items() if k != "matches"}}
        sm.close()
        if with_cpu:
            from oracle import karto_port as P
            pm = _port_matcher(grid, seq_mapper)
            exact, cpu = True, []
            for i, c in enumerate(cases):
                pq = P.PortScan(c["query_ranges"], c["query_pose"], synth.ANGLE_MIN, synth.ANGLE_INC)
                pb = [P.PortScan(r, p, synth.ANGLE_MIN, synth.ANGLE_INC) for r, p in zip(c["base_ranges"], c["base_poses"])]
                t = time.perf_counter()
                e = pm.match(pq, pb, True, True)
                cpu.append(1e3 * (time.perf_counter() - t))
                g = res[i]
                exact = exact and e[0] == g[0] and np.array_equal(e[1], g[1]) and np.array_equal(e[2], g[2])
            row.update({"cpu_ms_per_match_1core": float(np.mean(cpu)), "cpu_kind": "port (C restatement, pinned to the reference)",
                        "parity_exact": bool(exact), "speedup_vs_1core": float(np.mean(cpu)) / gpu_ms})
        out[tag] = row
    return out


def replay_bench(n_scans: int, n_ref: int):
    """cfg3: offline synchronous replay through the reference's own karto::Mapper::Process (integration/): GPU matcher (link-time
    seam) + GPU solver adapter on all n_scans; the reference CPU matcher on the first n_ref scans only (it runs ~20 scans/s), and the
    GPU path again on that same prefix for the identical-poses check."""
    sys.path.insert(0, os.path.join(ROOT, "integration"))
    import replay
    if not replay.available():
        return {"unavailable": "integration/_build/libreplay_*.so not built (needs the reference sources at build time)"}
    ranges, odom, _ = replay.make_trajectory(6, n_scans)
    params = dict(replay.YAML_PARAMS)
    out = {"workload": f"cfg3 replay: {n_scans} posed 1081-beam scans, slam_toolbox's shipped YAML parameters (smear 0.1 -> order-dependent "
                       f"raster, loop search 8 m), per-scan match + incremental graph build + solver after every loop closure"}

    def row(r):
        return {"scans_in": int(len(r["kept"])) if "kept" in r else None, "scans_kept": int(r["scans"]), "edges": int(r["edges"]),
                "process_s": float(r["process_seconds"]), "scans_per_s": float(r["scans"]) / float(r["process_seconds"]),
                "solver_computes": int(r["solver_computes"]), "solver_ms_total": float(r["solver_ms"]), "match_calls": int(r["match_calls"])}
    full = replay.run("b200", ranges, odom, params)
    out["b200_full"] = row(full)
    ref = replay.run("ref", ranges[:n_ref], odom[:n_ref], params)
    pre = replay.run("b200", ranges[:n_ref], odom[:n_ref], params)
    out["reference_prefix"] = dict(row(ref), scans_replayed=n_ref)
    out["b200_prefix"] = dict(row(pre), scans_replayed=n_ref)
    out["identical_poses_on_prefix"] = bool(np.array_equal(ref["poses"], pre["poses"]))
    out["speedup_on_prefix"] = out["b200_prefix"]["scans_per_s"] / out["reference_prefix"]["scans_per_s"]
    return out


def cfg5_bench(rank: int, world: int, stream, flush, n_query: int, n_cand: int, chain_len: int, steps: int):
    """cfg5: Q query scans x (n_cand x world) candidate chains, candidates sharded over the ranks, queries replicated.  One step =
    every rank sweeps its Q x n_cand pairs, builds its per-query winner records on the device and joins ONE all-gather; every rank
    then holds every query's winner.  Returns (device ms, e2e ms, pairs per rank) -- max over ranks is taken by the caller."""
    import torch
    import torch.distributed as dist
    from slam_toolbox_b200 import api, synth
    world_map = synth.make_world(7)
    rng = np.random.default_rng(2024)
    qtrue = synth.poses_near(world_map, synth.free_pose(world_map, rng)[:2], 2.0, n_query, rng)
    qr = synth.noisy(synth.raycast(world_map, qtrue), rng)
    qp = qtrue + np.column_stack([rng.normal(0, 0.4, (n_query, 2)), rng.normal(0, 0.06, n_query)])
    crng = np.random.default_rng(777 + rank)
    starts = synth.poses_near(world_map, qtrue[0, :2], 3.0, n_cand, crng)
    cp = starts if chain_len == 1 else np.concatenate([synth.chain_poses(world_map, st, chain_len, crng) for st in starts])
    cr = synth.noisy(synth.raycast(world_map, cp, chunk=64), crng)
    cs = np.arange(0, n_cand * chain_len + 1, chain_len, dtype=np.int32)
    laser = api.LaserRangeFinder()
    mapper = api.MapperParams(**{k: (bool(v) if k == "use_response_expansion" else v) for k, v in LOOP_MAPPER.items()})
    sm = api.ScanMatcher.Create(mapper, *LOOP_GRID)
    sm.set_stream(stream.cuda_stream)
    pts = torch.empty((cr.shape[0], cr.shape[1], 2), dtype=torch.float64).pin_memory()
    pts.numpy()[...] = api.point_readings(cr, cp, laser)
    cands, queries = api.ScanBlock(cr, cp, laser, points=pts.numpy()), api.ScanBlock(qr, qp, laser)
    rec_bytes = api.ScanMatcher.winner_record_bytes()
    send = torch.zeros(n_query * rec_bytes, dtype=torch.uint8, device="cuda")
    recv = torch.zeros(world * n_query * rec_bytes, dtype=torch.uint8, device="cuda")

    def exchange():
        sm.batch_winner_records(send.data_ptr(), rank * n_cand)
        if world > 1:
            dist.all_gather_into_tensor(recv, send)
        else:
            recv.copy_(send)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    npairs = sm.batch_upload(queries, cands, cs, None, False)
    sm.batch_run(); exchange()
    barrier()
    ev = []
    for k in range(steps):
        flush.fill_(k & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); sm.batch_run(); exchange(); b.record(stream)
        ev.append((a, b))
    barrier()
    dev_ms = float(np.sum([a.elapsed_time(b) for a, b in ev]))
    resp, _, _ = sm.batch_fetch()
    win = sm.batch_winners_select(recv.data_ptr(), world, n_query)
    sm.MatchScanBatch(queries, cands, cs, None, False, False)
    barrier()
    t = time.perf_counter()
    for _ in range(steps):
        r2 = sm.MatchScanBatch(queries, cands, cs, None, False, False)
        exchange()
        win = sm.batch_winners_select(recv.data_ptr(), world, n_query)
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t)
    # the winner every rank holds is the best candidate of its owner
    best = r2[0].reshape(n_query, n_cand)
    ok = True
    for q in range(n_query):
        if rank * n_cand <= win[0][q] < (rank + 1) * n_cand:
            ok = ok and win[1][q] == best[q].max() and int(win[0][q]) - rank * n_cand == int(np.argmax(best[q]))
        ok = ok and win[1][q] >= best[q].max()
    info = sm.batch_info()
    sm.close()
    return dev_ms, e2e_ms, npairs, bool(ok), info["kernel"], float(win[1].mean())


def graph_solve_case(sigma, steps: int, with_cpu: bool, peak_gbs: float, outputs: dict | None = None, tag: str = "graph"):
    """One cfg4 graph (10k nodes / 40k edges, dead-reckoned start) at one measurement-noise level, solved `steps` times on ONE
    solver handle (like the mapper's: device buffers persist, Reset + re-adding the graph makes every solve a cold graph).
    `outputs` receives the node ids and corrected poses of the last timed solve as <tag>_ids / <tag>_poses."""
    from slam_toolbox_b200 import synth, api
    g = synth.make_pose_graph(0, GRAPH_NODES, GRAPH_EDGES, sigma_xy=sigma[0], sigma_th=sigma[1])
    E = int(len(g["edge_a"]))
    out = {"nodes": GRAPH_NODES, "edges": E, "sigma_xy": sigma[0], "sigma_th": sigma[1], "init": "dead-reckoned odometry"}
    s = api.ScanSolver()
    rows, summ, poses, ok = [], None, None, False
    for i in range(steps + 1):   # first solve is the warm-up (allocations, cooperative-launch set-up)
        s.Reset()
        for nid, p in zip(g["ids"], g["init"]):
            s.AddNode(int(nid), p)
        for a, b, z, c in zip(g["edge_a"], g["edge_b"], g["z"], g["cov"]):
            s.AddConstraint(int(a), int(b), z, c)
        t = time.perf_counter()
        ok = s.Compute()
        wall = (time.perf_counter() - t) * 1e3
        summ = s.summary
        if i > 0:
            rows.append((summ.solve_ms, wall, summ.setup_ms))
        ids, poses = s.GetCorrections()
    if outputs is not None:
        outputs[f"{tag}_ids"], outputs[f"{tag}_poses"] = ids, poses
    ms = float(np.mean([r[0] for r in rows]))
    # what the mapper does after the NEXT loop closure (Mapper.cpp:2012-2030): one more constraint on the solved graph
    k = E - 1
    s.RemoveConstraint(int(g["edge_a"][k]), int(g["edge_b"][k]))
    s.Compute()
    s.AddConstraint(int(g["edge_a"][k]), int(g["edge_b"][k]), g["z"][k], g["cov"][k])
    t = time.perf_counter()
    s.Compute()
    inc_wall = (time.perf_counter() - t) * 1e3
    inc = {"wall_ms": inc_wall, "device_ms": float(s.summary.solve_ms), "uploaded_constraints": int(s.summary.uploaded_edges),
           "lm_iterations": int(s.summary.iterations), "what": "Compute after one constraint is appended to the solved graph"}
    s.close()
    # algorithmic bytes (SURVEY.md 8d): 584 B/edge per linearisation; per PCG iteration the block-sparse normal matrix
    # ((N + 2E) 3x3 FP64 blocks + column indices) and 5 vectors read + written
    lin_bytes = 584.0 * E
    pcg_bytes = (GRAPH_NODES + 2 * E) * (72 + 4) + 5 * 2 * GRAPH_NODES * 24
    n_lin = 2 + int(summ.iterations) + int(summ.successful_steps)
    total_bytes = n_lin * lin_bytes + int(summ.pcg_iterations) * pcg_bytes
    out.update({"ms": ms, "wall_ms": float(np.mean([r[1] for r in rows])), "host_setup_ms": float(np.mean([r[2] for r in rows])),
                "usable": bool(ok), "lm_iterations": int(summ.iterations), "successful_steps": int(summ.successful_steps),
                "pcg_iterations": int(summ.pcg_iterations), "final_cost": float(summ.final_cost),
                "kernel_launches": int(summ.kernel_launches), "incremental": inc,
                "roofline": {"bound": "hbm", "achieved": total_bytes / (ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                             "frac": total_bytes / (ms * 1e-3) / 1e9 / peak_gbs, "algorithmic_bytes": total_bytes,
                             "bytes_per_pcg_iteration": pcg_bytes, "bytes_per_linearisation": lin_bytes,
                             "us_per_pcg_iteration_incl_everything": 1e3 * ms / max(int(summ.pcg_iterations), 1),
                             "note": "the 15 MB problem is L2 resident: the solve is a chain of dependent block steps "
                                     "(latency x iterations), not HBM traffic; HBM is the mandated denominator"}})
    if with_cpu:
        from oracle import posegraph as PG
        t = time.perf_counter()
        xo, so = PG.solve(g["init"], g["edge_a"], g["edge_b"], g["z"], cov=g["cov"])
        cpu_ms = (time.perf_counter() - t) * 1e3
        d = poses - xo
        d[:, 2] = synth.wrap(d[:, 2])
        out["cpu_baseline"] = {"ms": cpu_ms, "kind": "port", "cores": 1,
                               "what": "python port, NOT Ceres: restated Ceres LM + SciPy SuperLU exact solves on one core (Ceres "
                                       "itself is not installable here; the reference README quotes <~0.3 s for graphs of a few "
                                       "thousand nodes with CHOLMOD)",
                               "lm_iterations": so.iterations, "successful_steps": so.successful_steps, "final_cost": so.final_cost}
        out["parity_vs_oracle"] = {"protocol": "P1: reference tolerances, same accept/reject sequence",
                                   "same_lm_iterations": bool(so.iterations == summ.iterations and so.successful_steps == summ.successful_steps),
                                   "max_abs_dxy_m": float(np.abs(d[:, :2]).max()), "max_abs_dtheta_rad": float(np.abs(d[:, 2]).max())}
    return out


def graph_solve_bench(steps: int, with_cpu: bool, peak_gbs: float = 6650.0, outputs: dict | None = None):
    """cfg4 at the contract's noise level (SURVEY.md 8d: 0.05 m / 0.02 rad) and at the lower one round 1 reported."""
    out = graph_solve_case((0.05, 0.02), steps, with_cpu, peak_gbs, outputs, "graph")
    out["low_noise_variant"] = graph_solve_case(GRAPH_SIGMA, steps, with_cpu, peak_gbs, outputs, "graph_low_noise")
    return out


def occupancy_bench(steps: int, with_cpu: bool, outputs: dict | None = None):
    """Map publish (SURVEY.md 8f row 4): OccupancyGrid::CreateFromScans over a cfg3-sized run of 5,000 scans at 0.05 m.
    `outputs` receives the grid of the last timed build: occupancy_cells, occupancy_passes, occupancy_hits."""
    from slam_toolbox_b200 import synth, api
    n_scans, res = 5000, 0.05
    run = synth.make_mapping_run(3, n_scans, world=synth.make_world(3, size=60.0), odd_readings=False)
    blk = api.ScanBlock(run["ranges"], run["poses"], api.LaserRangeFinder())
    g = api.OccupancyGrid(res, blk.laser)
    g.AddScans(blk)
    g.Build()                                    # warm-up: allocations
    ms = []
    for _ in range(steps):
        g.Build()
        ms.append(g.kernel_ms())
    cells, ps, ht = g.GetData(counters=True)
    if outputs is not None:
        outputs.update(occupancy_cells=cells, occupancy_passes=ps, occupancy_hits=ht)
    updates = int(ps.sum())
    launches = g.launch_count()
    g.close()
    e2e = []
    for _ in range(3):                           # through the public one-shot call: H2D of all scans + build + cells D2H
        t = time.perf_counter()
        g2 = api.OccupancyGrid.CreateFromScans(blk, res)
        c2 = g2.GetData()
        e2e.append((time.perf_counter() - t) * 1e3)
        g2.close()
    out = {"scans": n_scans, "beams": int(run["ranges"].size), "resolution": res, "grid": [int(cells.shape[1]), int(cells.shape[0])],
           "ms": float(np.mean(ms)), "scans_per_s": n_scans / (float(np.mean(ms)) * 1e-3), "cell_updates": updates,
           "cell_updates_per_s": updates / (float(np.mean(ms)) * 1e-3), "e2e_ms": float(min(e2e)),
           "h2d_bytes": int(run["ranges"].nbytes * 3 + run["poses"].shape[0] * 20), "d2h_bytes": int(cells.nbytes),
           "kernel_launches_per_build": 3, "kernel_launches": int(launches)}
    if with_cpu:
        from oracle import karto_ref as R, karto_port as P
        if R.available():
            R.init_laser(min_angle=synth.ANGLE_MIN, max_angle=synth.ANGLE_MAX, ang_res=synth.ANGLE_INC, min_range=0.1, max_range=30.0,
                         range_threshold=12.0)
            scans = [R.RefScan(r, p, i) for i, (r, p) in enumerate(zip(run["ranges"], run["poses"]))]
            ref = R.occupancy(scans, res)
            kind = "reference"
        else:
            scans = [P.PortScan(r, p, synth.ANGLE_MIN, synth.ANGLE_INC) for r, p in zip(run["ranges"], run["poses"])]
            ref = P.occupancy(scans, res, 12.0, 0.1, 30.0)
            kind = "port"
        out["cpu_baseline"] = {"ms": ref["seconds"] * 1e3, "kind": kind, "cores": 1,
                               "what": "OccupancyGrid::CreateFromScans on the same scans (single-threaded in the reference)"}
        out["parity_exact"] = bool(np.array_equal(ref["cells"], cells) and np.array_equal(ref["passes"], ps) and np.array_equal(ref["hits"], ht)
                                   and np.array_equal(c2, cells))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="skip the pose-graph solve part")
    ap.add_argument("--no-map", action="store_true", help="skip the occupancy-grid (map publish) part")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-rows", action="store_true", help="skip the extra sweep workloads (shipped geometries, chains, tie overflow)")
    ap.add_argument("--no-seq", action="store_true", help="skip the cfg1 sequential-match section")
    ap.add_argument("--no-replay", action="store_true", help="skip the cfg3 replay section")
    ap.add_argument("--replay-scans", type=int, default=5000)
    ap.add_argument("--replay-ref-scans", type=int, default=400)
    ap.add_argument("--sweep-kernel", type=int, default=0, help="0 auto, 1 single-CTA kernel, 2 tiled cluster kernel (headline workload)")
    ap.add_argument("--chain-len", type=int, default=CHAIN_LEN)
    ap.add_argument("--candidates", type=int, default=N_CAND)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step as DIR/<name>.npy: "
                    "the headline sweep's response, mean and covariance per pair (rank 0's shard), and the pose-graph poses and "
                    "occupancy grid when those parts run")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from slam_toolbox_b200 import api, sweep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the b200 implementation has no CPU fallback")
    torch.cuda.set_device(local_rank)
    api._check(api.lib().b200_set_device(local_rank))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))

    n_cand, chain_len = args.candidates, args.chain_len
    qr, qp, cr, cp, cs = make_inputs(rank, n_cand, chain_len, N_QUERY)
    laser = api.LaserRangeFinder()
    mapper = api.MapperParams(**{k: (bool(v) if k == "use_response_expansion" else v) for k, v in LOOP_MAPPER.items()})
    sm = api.ScanMatcher.Create(mapper, *LOOP_GRID)
    sm.set_option("sweep_kernel", args.sweep_kernel)
    stream = torch.cuda.Stream()          # a real (non-default) stream shared by torch and the library
    torch.cuda.set_stream(stream)
    sm.set_stream(stream.cuda_stream)

    # host inputs in pinned memory (the e2e leg copies from here every step)
    pts_pinned = torch.empty((cr.shape[0], cr.shape[1], 2), dtype=torch.float64).pin_memory()
    pts_np = pts_pinned.numpy()
    pts_np[...] = api.point_readings(cr, cp, laser)
    cands = api.ScanBlock(cr, cp, laser, points=pts_np)
    assert cands.points.ctypes.data == pts_np.ctypes.data
    queries = api.ScanBlock(qr, qp, laser)
    npairs = N_QUERY * n_cand
    keys = torch.zeros(N_QUERY, dtype=torch.int64, device="cuda")
    pair_q = np.repeat(np.arange(N_QUERY), n_cand)                       # pairs are query-major when no pair list is given
    pair_c_global = np.tile(np.arange(n_cand), N_QUERY) + rank * n_cand
    winners = None
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wx = sweep.WinnerExchange(sm, N_QUERY, world)

    def exchange():
        """the multi-GPU step: this rank's best candidate per query (device kernel) -> ONE all-gather over NVLink -> every rank
        selects the same winner; no host round trip before the collective"""
        wx.gather(rank * n_cand)

    def device_step():
        sm.batch_run()
        if world > 1:
            exchange()

    # ---- device-resident leg: inputs uploaded once ----
    sm.batch_upload(queries, cands, cs, None, False)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        device_step()
    barrier()
    if rank == 0:
        sampler.wait_first()
    launches0 = sm.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []
    barrier()
    t_wall = time.perf_counter()
    for k in range(args.steps):
        flush.fill_(k & 0xFF)            # evict L2 between timed iterations (outside the event pair)
        ev[k][0].record(stream)
        device_step()
        ev[k][1].record(stream)
        kernel_ms.append(None)
    barrier()
    t_wall = time.perf_counter() - t_wall
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = float(np.sum(step_ms))
    last_kernel_ms = sm.batch_kernel_ms()
    launches = sm.launch_count() - launches0
    resp_dev, mean_dev, cov_dev = sm.batch_fetch()
    clocks = sampler.stop() if rank == 0 else None

    # ---- end-to-end leg: public API, host inputs, copies inside the timed region ----
    sm.transfer_bytes(reset=True)
    for _ in range(2):
        r_e2e = sm.MatchScanBatch(queries, cands, cs, None, False, False)
        if world > 1:
            exchange()
            winners = wx.select()
    sm.transfer_bytes(reset=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r_e2e = sm.MatchScanBatch(queries, cands, cs, None, False, False)
        if world > 1:
            exchange()
            winners = wx.select()
    barrier()
    e2e_s = time.perf_counter() - t0
    h2d, d2h = sm.transfer_bytes()
    assert np.array_equal(r_e2e[0], resp_dev)
    if world > 1:   # every rank holds the same winner rows, and the owner's row is its own result
        gid = winners[0]
        for q in range(N_QUERY):
            if rank * n_cand <= gid[q] < (rank + 1) * n_cand:
                j = q * n_cand + int(gid[q]) - rank * n_cand
                assert winners[1][q] == r_e2e[0][j] and np.array_equal(winners[2][q], r_e2e[1][j]) and np.array_equal(winners[3][q], r_e2e[2][j])
                assert r_e2e[0][j] == r_e2e[0][q * n_cand:(q + 1) * n_cand].max()

    # max over ranks
    t = torch.tensor([dev_ms, e2e_s * 1e3, last_kernel_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, kern_ms = [float(v) for v in t.tolist()]
    total_pairs = npairs * world
    value = total_pairs * args.steps / (dev_ms * 1e-3)
    e2e_value = total_pairs * args.steps / (e2e_ms * 1e-3)

    cfg5 = None
    if world > 1 and not args.no_rows:
        rows5 = []
        for label, nq5, nc5, cl5 in (("chain length 1", 32, 6250, 1), ("chain length 10", 32, 625, 10)):
            dms, ems, np5, ok5, kern5, mean_best = cfg5_bench(rank, world, stream, flush, nq5, nc5, cl5, 2)
            t5 = torch.tensor([dms, ems], dtype=torch.float64, device="cuda")
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
            okt = torch.tensor([1 if ok5 else 0], dtype=torch.int32, device="cuda")
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            dms, ems = [float(v) for v in t5.tolist()]
            tot = np5 * world * 2
            rows5.append({"variant": label, "queries": nq5, "candidate_chains_per_gpu": nc5, "candidate_chains_total": nc5 * world,
                          "pairs_per_step": np5 * world, "value": tot / (dms * 1e-3), "unit": UNIT, "ms_per_step": dms / 2,
                          "e2e": {"value": tot / (ems * 1e-3), "ms_per_step": ems / 2}, "kernel": kern5,
                          "winners_consistent_on_every_rank": bool(int(okt.item())), "mean_winning_response": mean_best,
                          "full_cfg5_seconds_at_this_rate": 256 * 50000 / (tot / (dms * 1e-3))})
        cfg5 = {"what": "cfg5 (256 queries x 50,000 candidates over 8 GPUs) as a time-bounded sample: 32 of the 256 queries against the "
                        "full 6,250 candidate chains per GPU (chain length 10: 625 chains per GPU); candidates sharded, queries replicated, "
                        "one all_gather of the winner records per step", "rows": rows5}
    if rank != 0:
        if world > 1:
            dist.barrier()   # rank 0 finishes the CPU baseline / graph solve, then everyone leaves together
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the fused sweep kernel) ----
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    n_angles = int(math.floor(2 * LOOP_MAPPER["coarse_search_angle_offset"] / LOOP_MAPPER["coarse_angle_resolution"] + 0.5)) + 1
    bytes_per_launch = algorithmic_bytes_per_match(cr.shape[1], n_angles, npairs, N_QUERY) * npairs
    achieved = bytes_per_launch / (kern_ms * 1e-3) / 1e9
    gathers = npairs * 41 * 41 * n_angles * cr.shape[1]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "peak_source": peak_src, "kernel": {"tile": "k_sweep_tile (tiled cluster kernel: raster + correlation + distributed reduction)", "fast": "k_sweep_fast",
                           "generic": "k_sweep_generic"}[sm.batch_info()["kernel"]], "kernel_ms": kern_ms,
                "algorithmic_bytes_per_match": bytes_per_launch / npairs,
                "onchip": {"gathers_per_s": gathers / (kern_ms * 1e-3), "smem_gather_ceiling_per_s": 32 * 148 * 1.9e9,
                           "frac_of_128B_per_clk_per_SM": gathers / (kern_ms * 1e-3) / (128 * 148 * 1.965e9),
                           "note": "the path is bound by on-chip gather/ALU issue rate, not HBM (SURVEY.md 7.5)"}}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            roofline["traffic"] = json.load(open(prof)).get("sweep_kernel_dram_bytes_per_launch")
        except Exception:
            pass

    # ---- CPU baseline on the host cores (bounded sample of the same workload) ----
    cpu = None
    if not args.no_cpu:
        threads = host_threads()
        n_sample = min(n_cand, max(16, 12 * min(threads, 32)))
        rate, kind, sec, resp_cpu, used = cpu_sweep(qr, qp, cr, cp, cs, n_sample, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": used, "kind": kind, "host_threads_available": threads,
               "sample": f"first {n_sample} of {n_cand} candidate matches, one reference ScanMatcher per host thread "
                         f"({used} threads: the fastest of the counts tried), {sec:.2f} s",
               "parity_exact": bool(np.array_equal(resp_cpu, resp_dev[:n_sample]))}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": f"cfg2 loop-closure batch: {N_QUERY} query x {n_cand} candidate chains (chain length {chain_len}) of "
                               f"1081-beam scans per GPU, +-2m/+-20deg window, candidates sharded over {world} GPU(s)",
                   "search": f"41x41x{n_angles} poses", "grid": "565x568 u8 (res 0.05 m, smear 0.03 m, range threshold 12 m)",
                   "l2": "L2 flushed between timed steps (256 MiB write)", "collective": "one all_gather of the per-query winner records (152 B per query and rank), winners selected locally on every rank" if world > 1 else "none",
                   "kernel": sm.batch_info()["kernel"]},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d // args.steps, "d2h_bytes_per_step": d2h // args.steps,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "wall_ms_per_step_incl_flush": 1e3 * t_wall / args.steps,
    }
    if cfg5 is not None:
        line["cfg5"] = cfg5
    if world == 1 and not args.no_rows:
        k = max(3, min(args.steps, 5))
        dim8, rt20, both = (8.0, 0.05, 0.03, 12.0), (4.0, 0.05, 0.03, 20.0), (8.0, 0.05, 0.03, 20.0)
        line["sweep_rows"] = [
            sweep_row("cfg2 on round 1's single-CTA kernel (k_sweep_fast) for comparison; the headline runs the tiled cluster kernel", LOOP_GRID, 1000, 1, k, peak, stream, flush, {"sweep_kernel": 1}),
            sweep_row("loop_search_space_dimension 8 m (toolbox / Karto default, mapper_params_online_sync.yaml:61), rt 12 m", dim8, 1000, 1, k, peak, stream, flush),
            sweep_row("max_laser_range 20 m (mapper_params_online_sync.yaml:32), search 4 m", rt20, 1000, 1, k, peak, stream, flush),
            sweep_row("shipped YAML geometry: search 8 m + range threshold 20 m", both, 1000, 1, k, peak, stream, flush),
            sweep_row("cfg2 with chains of 10 scans (loop_match_minimum_chain_size, Mapper.cpp:2001)", LOOP_GRID, 1000, 10, k, peak, stream, flush),
            sweep_row("cfg2 with 50 % of the candidates not overlapping the query (all poses tie at 0: closed form, no per-pair fall back)", LOOP_GRID, 1000, 1, k, peak, stream, flush, far_fraction=0.5),
            sweep_row("small batch, one pair per 8-CTA cluster (latency mode): 8 candidate chains of 10 scans, search 8 m", dim8, 8, 10, k, peak, stream, flush, {"sweep_kernel": 2, "sweep_cluster": 8}, parity_samples=2),
            sweep_row("the same small batch on one CTA per pair", dim8, 8, 10, k, peak, stream, flush, {"sweep_kernel": 2, "sweep_cluster": 1}, parity_samples=2),
            sweep_row("cfg5 shape on one GPU: 16 queries x 6,250 candidates", LOOP_GRID, 6250, 1, 3, peak, stream, flush, n_query=16),
        ]
    if world == 1 and not args.no_seq:
        line["seq_match"] = seq_match_bench(200, not args.no_cpu)
    if world == 1 and not args.no_replay:
        try:
            line["replay"] = replay_bench(args.replay_scans, args.replay_ref_scans)
        except Exception as ex:   # the replay needs the prebuilt integration libraries
            line["replay"] = {"unavailable": str(ex)[-300:]}
    outputs = {"response": resp_dev, "mean": mean_dev, "covariance": cov_dev}
    if not args.no_graph:
        line["graph_solve"] = graph_solve_bench(3, not args.no_cpu, peak, outputs)
    if not args.no_map:
        line["occupancy_grid"] = occupancy_bench(5, not args.no_cpu, outputs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
