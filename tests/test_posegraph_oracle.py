"""Checks of the restated pose-graph oracle (oracle/posegraph.py; PARITY UNPINNED -- the reference's solver is
Ceres, which the tests do not link): its building blocks against the reference's own karto code where that exists
(LinkInfo, Matrix3::Inverse, through tests/golden/reference_posegraph_golden.npz) and its minimiser against
scipy.optimize.least_squares."""
import os

import numpy as np
import pytest
from scipy.optimize import least_squares

from oracle import posegraph as PG
from slam_toolbox_b200 import synth

REF_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_posegraph_golden.npz")


def test_normalize_angle_range():
    a = np.linspace(-20, 20, 1001)
    w = PG.normalize_angle(a)
    assert np.all(w >= -np.pi) and np.all(w < np.pi)
    assert np.allclose(np.sin(w), np.sin(a)) and np.allclose(np.cos(w), np.cos(a))
    assert PG.normalize_angle(np.array([np.pi]))[0] == -np.pi


def test_link_info_and_inverse_match_karto():
    z = np.load(REF_GOLDEN)
    assert len(z["p1"]) == 20
    for p1, p2, cov, d_ref, c_ref, inv_ref in zip(z["p1"], z["p2"], z["cov"], z["link_delta"], z["link_cov"], z["inverse"]):
        d, c = PG.link_info(p1, p2, cov)
        assert np.allclose(d[:2], d_ref[:2], atol=1e-12)
        assert abs(np.sin(d[2] - d_ref[2])) < 1e-12 and np.cos(d[2] - d_ref[2]) > 0
        assert np.allclose(c, c_ref, atol=1e-12)
        assert np.allclose(PG.matrix3_inverse(cov), inv_ref, rtol=1e-13, atol=0)


def test_sqrt_information_is_upper_cholesky_of_the_information():
    rng = np.random.default_rng(1)
    A = rng.normal(size=(3, 3))
    cov = A @ A.T + 0.5 * np.eye(3)
    U = PG.sqrt_information(cov)
    assert np.allclose(np.tril(U, -1), 0)
    assert np.allclose(U.T @ U, np.linalg.inv(cov), rtol=1e-10)


def test_jacobian_matches_finite_differences():
    g = synth.make_pose_graph(2, 40, 70, sigma_xy=0.03, sigma_th=0.01)
    U = np.stack([PG.sqrt_information(c) for c in g["cov"]])
    pb = PG.Problem(g["init"], g["edge_a"], g["edge_b"], g["z"], U, 0)
    x = g["init"].copy()
    J = pb.jacobian(x).toarray()
    r0 = pb.residuals(x)
    eps = 1e-6
    for k in range(0, J.shape[1], 7):
        d = np.zeros(J.shape[1]); d[k] = eps
        num = (pb.residuals(pb.plus(x, d)) - r0) / eps
        assert np.allclose(num, J[:, k], atol=2e-4 * (1 + np.abs(J[:, k]).max()))


@pytest.mark.parametrize("seed", [0, 1])
def test_lm_reaches_the_least_squares_minimiser(seed):
    g = synth.make_pose_graph(seed, 150, 400, sigma_xy=0.03, sigma_th=0.01)
    tight = PG.Options(function_tolerance=1e-15, parameter_tolerance=1e-14, gradient_tolerance=1e-14, max_num_iterations=200)
    x, sm = PG.solve(g["init"], g["edge_a"], g["edge_b"], g["z"], cov=g["cov"], opts=tight)
    assert sm.usable
    U = np.stack([PG.sqrt_information(c) for c in g["cov"]])
    pb = PG.Problem(g["init"], g["edge_a"], g["edge_b"], g["z"], U, 0)

    def fun(p):
        xx = x.copy()
        xx[pb.free] = p.reshape(-1, 3)
        return pb.residuals(xx)

    ref = least_squares(fun, x[pb.free].reshape(-1), method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    xr = x.copy()
    xr[pb.free] = ref.x.reshape(-1, 3)
    d = xr - x
    d[:, 2] = synth.wrap(d[:, 2])
    assert np.abs(d).max() < 1e-6
    assert abs(0.5 * float(ref.fun @ ref.fun) - sm.final_cost) < 1e-9 * max(1.0, sm.final_cost)
    # anchor untouched; cost decreased
    assert np.array_equal(x[0], g["init"][0]) and sm.final_cost < sm.initial_cost


def test_reference_tolerances_stop_early_but_near_the_minimum():
    g = synth.make_pose_graph(3, 300, 800, sigma_xy=0.03, sigma_th=0.01)
    x, sm = PG.solve(g["init"], g["edge_a"], g["edge_b"], g["z"], cov=g["cov"])
    assert sm.usable and sm.iterations <= 50 and "CONVERGENCE" in sm.termination
    tight = PG.Options(function_tolerance=1e-15, parameter_tolerance=1e-14, gradient_tolerance=1e-14, max_num_iterations=200)
    _, st = PG.solve(g["init"], g["edge_a"], g["edge_b"], g["z"], cov=g["cov"], opts=tight)
    # function_tolerance 1e-3 stops close to the minimum cost, never below it
    assert st.final_cost <= sm.final_cost <= 1.25 * st.final_cost


def test_nodes_without_edges_and_missing_anchor_edges():
    g = synth.make_pose_graph(4, 30, 40, sigma_xy=0.03, sigma_th=0.01)
    init = np.vstack([g["init"], [[100.0, 100.0, 1.0]]])   # an isolated node: not a Ceres parameter block
    x, sm = PG.solve(init, g["edge_a"], g["edge_b"], g["z"], cov=g["cov"])
    assert np.array_equal(x[-1], init[-1]) and sm.usable
