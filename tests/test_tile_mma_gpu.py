"""The integer tensor-core beam loop of the tiled sweep kernel (csrc/sm_tile.cu): beams that share a cell become one entry whose
weight is their count (split above 255), one stream per (angle, stage) serves every byte alignment, k-quads are padded to
distinct word residues, and the accumulators are flushed once per warp item.  Each case is bit-exact against the oracle (C
restatement pinned to the reference) and against the generic kernel."""
from __future__ import annotations

import numpy as np
import pytest

from slam_toolbox_b200 import api, synth
import helpers as H

pytestmark = pytest.mark.gpu

MAPPER = dict(H.MAPPER_LOOP, use_response_expansion=0)


def _laser(min_angle, res, n, rt):
    return api.LaserRangeFinder(minimum_angle=min_angle, maximum_angle=min_angle + res * (n - 1), angular_resolution=res,
                                minimum_range=H.LASER["min_range"], maximum_range=H.LASER["max_range"], range_threshold=rt)


def _check(grid, qr, qp, cr, cp, chain_start, min_angle=synth.ANGLE_MIN, res=synth.ANGLE_INC, options=()):
    """Runs the sweep on the tiled kernel (automatic plan and two forced ones) and on the generic kernel, checks both against
    the oracle; returns the tiled kernel's batch_info."""
    from oracle import karto_port as P
    nq, nch = len(qr), len(chain_start) - 1
    pm, gm = H.port_matcher(MAPPER, grid), H.gpu_matcher(MAPPER, grid)
    pq = [P.PortScan(r, p, min_angle, res) for r, p in zip(qr, qp)]
    pc = [P.PortScan(r, p, min_angle, res) for r, p in zip(cr, cp)]
    exp = [pm.match(pq[q], pc[chain_start[c]:chain_start[c + 1]], False, False) for q in range(nq) for c in range(nch)]
    er, em, ec = (np.array([e[i] for e in exp]) for i in range(3))
    laser = _laser(min_angle, res, qr.shape[1], grid[3])
    gq, gc = api.ScanBlock(qr, qp, laser), api.ScanBlock(cr, cp, laser)
    for k, v in options:
        gm.set_option(k, v)
    gm.set_option("force_generic_sweep", 1)
    gen = gm.MatchScanBatch(gq, gc, chain_start, None, False, False)
    gen_best = gm.batch_best()
    assert np.array_equal(gen[0], er) and np.array_equal(gen[1], em) and np.array_equal(gen[2], ec)
    gm.set_option("force_generic_sweep", 0)
    gm.set_option("sweep_kernel", 2)
    info = None
    for cluster, chunks in ((0, 0), (1, 0), (2, 5)):
        gm.set_option("sweep_cluster", cluster)
        gm.set_option("sweep_chunks", chunks)
        r, m, c = gm.MatchScanBatch(gq, gc, chain_start, None, False, False)
        info, plan = gm.batch_info(), gm.batch_tile_info()
        assert info["kernel"] == "tile" and plan["available"], (info, plan)
        assert np.array_equal(r, er), (plan, r, er)
        assert np.array_equal(m, em) and np.array_equal(c, ec), plan
        for a, b in zip(gm.batch_best(), gen_best):   # best integer sum, arg-max pose index, tie count
            assert np.array_equal(a, b), plan
    return info


def _sweep(seed, nq=1, nch=6):
    sw = synth.make_loop_sweep(seed, n_queries=nq, n_chains=nch, chain_len=1)
    return sw.query_ranges, sw.query_poses, sw.cand_ranges, sw.cand_poses, sw.chain_start


def test_short_ranges_largest_weights():
    """Every query beam 0.1 .. 0.13 m from the sensor: up to ~115 beams of the 0.25 deg laser share one 5 cm cell."""
    qr, qp, cr, cp, cs = _sweep(51)
    rng = np.random.default_rng(51)
    qr = 0.101 + 0.03 * rng.random(qr.shape)
    cr = np.where(rng.random(cr.shape) < 0.5, cr, 0.101 + 0.03 * rng.random(cr.shape))
    _check(H.GRID_LOOP, qr, qp, cr, cp, cs)


def test_weight_above_255_splits():
    """A laser of 1e-4 rad steps whose returns alternate between 0.11 m and 0.26 m: the 1201 near returns span a 2.9 cm arc, so
    at most 4 cells hold them and one cell takes more than 255 beams of every search angle -- its weight is split over several
    entries of the same word.  The far returns keep consecutive points more than 0.1 m apart, so FindValidPoints keeps the
    candidates' points and the raster is not empty."""
    n, res, a0 = 2401, 1e-4, -0.12
    rng = np.random.default_rng(52)

    def zigzag(rows):
        r = np.empty((rows, n))
        r[:, 0::2] = 0.11 + 0.002 * rng.random((rows, (n + 1) // 2))
        r[:, 1::2] = 0.26 + 0.002 * rng.random((rows, n // 2))
        return r

    qr, qp = zigzag(1), np.array([[0.3, -0.2, 0.05]])
    cp = qp + np.column_stack([rng.normal(0, 0.05, (4, 2)), rng.normal(0, 0.02, 4)])
    cr = zigzag(4)
    assert 0.112 * res * (n - 1) < 0.05 and (n + 1) // 2 > 4 * 255   # near arc inside 2 x 2 cells, more than 4 x 255 beams
    grid = (1.0, 0.05, 0.03, 6.0)
    from oracle import karto_port as P
    pm = H.port_matcher(MAPPER, grid)
    q = P.PortScan(qr[0], qp[0], a0, res)
    for j in range(4):
        c = P.PortScan(cr[j], cp[j], a0, res)
        assert len(P.find_valid_points(c, cp[j][:2])) > n // 2
        assert pm.match(q, [c], False, False)[0] > 0.0   # the dense cells meet rastered cells under some search pose
    _check(grid, qr, qp, cr, cp, np.arange(5, dtype=np.int32), min_angle=a0, res=res)


@pytest.mark.parametrize("grid,seed", [((0.5, 0.05, 0.03, 6.0), 53), ((0.3, 0.05, 0.03, 5.0), 54), ((1.1, 0.05, 0.04, 7.0), 55),
                                       ((1.4, 0.05, 0.03, 7.5), 56), ((2.6, 0.05, 0.03, 9.0), 57), ((0.9, 0.05, 0.03, 4.5), 60)])
def test_small_and_odd_windows(grid, seed):
    """Coarse windows of 4 .. 27 poses a side (every residue of the width mod 4): every byte alignment, streams of a few steps
    padded to distinct residues, word ranges with unused slots."""
    _check(grid, *_sweep(seed, nq=2, nch=4))


def test_no_beam_dedup_on_tile_kernel():
    """no_beam_dedup: every beam is its own weight-1 entry."""
    qr, qp, cr, cp, cs = _sweep(58)
    qr = np.minimum(qr, 0.6)
    _check(H.GRID_LOOP, qr, qp, cr, cp, cs, options=(("no_beam_dedup", 1),))


def test_edge_beams_with_6m_threshold():
    """A 6 m range threshold shrinks the grid so that some beams' windows leave it (EDGE path next to the tensor-core path)."""
    info = _check((4.0, 0.05, 0.03, 6.0), *_sweep(59, nq=1, nch=6))
    assert info["edge_beams"] > 0, info
