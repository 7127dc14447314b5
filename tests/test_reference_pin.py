"""The oracle (and, on the GPU, the CUDA path) against outputs of the REFERENCE'S OWN SCRIPTS.

tests/golden/reference_run.json was written by tests/golden/make_golden_from_reference.py, which executed the
reference's arbitrage.py, liquidation.py and two-asset.py unmodified (runpy) with oracle/cvxpy_shim.py standing in for
the absent cvxpy.  The fixture holds what the scripts read back after prob.solve(): prob.value, psi.value,
deltas[i].value, lambdas[i].value (arbitrage.py:84, liquidation.py:87) and, per swept amount t, obj.value and
lambdas[k].value - deltas[k].value (two-asset.py:93-100)."""
import json
import os

import numpy as np
import pytest

from cfmm_routing_code_b200 import instances as I
from oracle import cfmm_oracle as O
from oracle import cvxpy_shim as cp
import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref_run():
    with open(os.path.join(ROOT, "tests", "golden", "reference_run.json")) as f:
        return json.load(f)


def test_instances_restate_the_reference_literals_exactly(ref_run):
    """cfmm_routing_code_b200.instances vs the literals the executed scripts defined (arbitrage.py:5-36 etc.)"""
    for name, d in (("arbitrage", I.arbitrage_instance()), ("liquidation", I.liquidation_instance()),
                    ("two_asset", I.two_asset_instance())):
        g = ref_run[name]["data"]
        assert d["n_tokens"] == g["n_tokens"] and d["local_indices"] == g["local_indices"]
        assert [list(map(float, r)) for r in d["reserves"]] == g["reserves"]
        assert [float(f) for f in d["fees"]] == g["fees"]
    assert [float(v) for v in I.arbitrage_instance()["market_value"]] == ref_run["arbitrage"]["data"]["market_value"]
    assert [float(v) for v in I.liquidation_instance()["current_assets"]] == ref_run["liquidation"]["data"]["current_assets"]
    assert np.array_equal(I.two_asset_instance()["amounts"], np.asarray(ref_run["two_asset"]["amounts"]))


def test_oracle_matches_the_executed_reference_scripts(ref_run):
    d = I.arbitrage_instance(); g = ref_run["arbitrage"]
    assert g["status"] == "optimal"
    r = O.solve(H.oracle_pools(H.host_pools(d)), O.Utility.arbitrage(d["market_value"]), tol=1e-10)
    assert r.status == "optimal" and abs(r.value - g["value"]) <= 1e-8 * abs(g["value"])
    np.testing.assert_allclose(r.psi, g["psi"], atol=2e-6)
    for i in range(5):
        np.testing.assert_allclose(r.deltas[i], g["deltas"][i], atol=5e-5)
        np.testing.assert_allclose(r.lambdas[i], g["lambdas"][i], atol=5e-5)
    d = I.liquidation_instance(); g = ref_run["liquidation"]
    r = O.solve(H.oracle_pools(H.host_pools(d)), O.Utility.liquidate(5, d["target"], d["current_assets"]), tol=1e-10)
    assert r.status == "optimal" and abs(r.value - g["value"]) <= 1e-8 * abs(g["value"])
    np.testing.assert_allclose(r.psi, g["psi"], atol=2e-6)
    for i in range(5):
        np.testing.assert_allclose(r.deltas[i], g["deltas"][i], atol=5e-5)
        np.testing.assert_allclose(r.lambdas[i], g["lambdas"][i], atol=5e-5)
    d = I.two_asset_instance(); g = ref_run["two_asset"]
    P = H.oracle_pools(H.host_pools(d))
    for j in range(50):
        r = O.solve(P, O.Utility.swap(3, 0, 2, d["amounts"][j]), tol=1e-10)
        assert abs(r.value - g["u_t"][j]) <= 1e-7 * max(abs(g["u_t"][j]), 1.0), j
        for k in range(5):          # two-asset.py:93-94: lambdas[k].value - deltas[k].value
            np.testing.assert_allclose(r.lambdas[k] - r.deltas[k], g["flows"][j][k], atol=5e-5, err_msg=f"t index {j}, pool {k}")


def test_reference_values_agree_with_the_zero_gap_certified_ones(ref_run, golden):
    """three derivations of the same optimum: the executed reference scripts, the restated primal (round 1 fixture) and
    SURVEY.md section 8c's zero-duality-gap values"""
    assert abs(ref_run["arbitrage"]["value"] - golden["survey_8c"]["arbitrage"]) <= 1e-9 * 21.5
    assert abs(ref_run["liquidation"]["value"] - golden["survey_8c"]["liquidation"]) <= 1e-9 * 15.9
    assert abs(ref_run["two_asset"]["u_t"][0] - golden["survey_8c"]["two_asset_t0"]) <= 1e-8
    assert abs(ref_run["two_asset"]["u_t"][49] - golden["survey_8c"]["two_asset_t50"]) <= 1e-8
    for j in range(50):
        assert abs(ref_run["two_asset"]["u_t"][j] - golden["two_asset"][j]["value"]) <= 1e-7 * max(1.0, golden["two_asset"][j]["value"])


def test_fixture_is_what_the_shim_computes_for_the_reference_problems(ref_run):
    """tests/routing_script.py (the three problems of the reference's scripts, stated with cvxpy's API) executed the way
    the fixture's generator executed the reference's scripts, with the shim standing in for cvxpy"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mk", os.path.join(ROOT, "tests", "golden", "make_golden_from_reference.py"))
    mk = importlib.util.module_from_spec(spec); spec.loader.exec_module(mk)
    g = mk.run_reference_script(os.path.join(ROOT, "tests", "routing_script.py"))
    assert abs(g["prob"].value - ref_run["arbitrage"]["value"]) <= 1e-10
    assert "Total output value" in g["__stdout__"]
    assert abs(g["liq_psi"].value[4] - ref_run["liquidation"]["value"]) <= 1e-10
    np.testing.assert_allclose(g["u_t"], ref_run["two_asset"]["u_t"], rtol=0, atol=1e-10)


def test_shim_models_what_cvxpy_would():
    """the cvxpy subset the scripts use, on programs with known answers"""
    x = cp.Variable(2, nonneg=True)
    A = np.array([[1.0, 0.0], [0.0, 1.0], [1.0, 1.0]])
    e = A @ x
    assert e.shape == (3,) and (np.array([1.0, 2.0, 3.0]) @ e).shape == ()
    # max x0 + x1 s.t. geo_mean(x) >= 1 is unbounded without a cap: add x <= 4 via 4 - x >= 0; optimum at (4, 4)
    p = cp.Problem(cp.Maximize(cp.sum(x)), [cp.geo_mean(x) >= 1.0, 4 - x >= 0])
    assert abs(p.solve() - 8.0) <= 1e-9 and p.status == "optimal"
    # min x0 + 2 x1 s.t. x0^(2/3) x1^(1/3) >= 1: Lagrange gives x0 = 2^(2/3) ... check against the closed form
    y = cp.Variable(2, nonneg=True)
    p = cp.Problem(cp.Minimize(np.array([1.0, 2.0]) @ y), [cp.geo_mean(y, p=np.array([2, 1])) >= 1.0])
    v = p.solve()
    w = np.array([2 / 3, 1 / 3]); c = np.array([1.0, 2.0])
    yy = (w / c) / np.prod((w / c) ** w)                      # x_j = (w_j / c_j) * t with prod x^w = 1
    assert abs(v - c @ yy) <= 1e-8 and np.allclose(y.value, yy, atol=1e-6)
    # equality and indexing
    z = cp.Variable(3, nonneg=True)
    p = cp.Problem(cp.Maximize(z[2]), [z[0] + 1.0 == 3.0, cp.sum(z) <= 10, z[1] >= 0.5])
    assert abs(p.solve() - 7.5) <= 1e-9 and abs(z.value[0] - 2.0) <= 1e-9
    assert cp.geo_mean(np.array([4.0, 4, 4, 4])) == pytest.approx(4.0)
    # infeasible
    q = cp.Variable(1, nonneg=True)
    p = cp.Problem(cp.Maximize(q[0]), [q[0] + 1.0 == 0.0])
    p.solve()
    assert p.status == "infeasible"


@pytest.mark.gpu
def test_cuda_path_matches_the_executed_reference_scripts(ref_run):
    """prob.solve() replaced by the CUDA path (through the C ABI), checked against what the reference's scripts produced"""
    import cfmm_routing_code_b200 as cf
    for method in ("pools", "thread"):
        d = I.arbitrage_instance(); g = ref_run["arbitrage"]
        r = cf.solve(d["local_indices"], d["reserves"], d["fees"], d["kinds"], d["weights"],
                     utility=cf.Arbitrage(d["market_value"]), tol=1e-9, method=method)
        assert r.status == "optimal" and abs(r.value - g["value"]) <= 1e-6 * abs(g["value"])     # north star: 1e-6 relative
        assert abs(r.value - g["value"]) <= 1e-8 * abs(g["value"])
        np.testing.assert_allclose(r.psi, g["psi"], atol=1e-6 * np.abs(g["psi"]).max())
        for i in range(5):
            np.testing.assert_allclose(r.deltas[i], g["deltas"][i], atol=5e-5)
            np.testing.assert_allclose(r.lambdas[i], g["lambdas"][i], atol=5e-5)
        d = I.liquidation_instance(); g = ref_run["liquidation"]
        r = cf.solve(d["local_indices"], d["reserves"], d["fees"], d["kinds"], d["weights"],
                     utility=cf.Liquidate(d["target"], d["current_assets"]), tol=1e-9, method=method)
        assert r.status == "optimal" and abs(r.psi[4] - g["value"]) <= 1e-8 * g["value"]
        np.testing.assert_allclose(r.psi, g["psi"], atol=1e-6 * np.abs(g["psi"]).max())
    d = I.two_asset_instance(); g = ref_run["two_asset"]
    rs = cf.solve_sweep(d["local_indices"], d["reserves"], d["fees"], d["kinds"], d["weights"],
                        [cf.Swap(d["tok_in"], d["tok_out"], t) for t in d["amounts"]], tol=1e-9)
    for j, r in enumerate(rs):
        assert r.status == "optimal" and abs(r.value - g["u_t"][j]) <= 1e-6 * max(1.0, g["u_t"][j]), j
        for k in range(5):
            np.testing.assert_allclose(r.lambdas[k] - r.deltas[k], g["flows"][j][k], atol=5e-5)
