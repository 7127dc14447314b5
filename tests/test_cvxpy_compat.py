"""`cfmm_routing_code_b200.cvxpy_compat`: the reference's cvxpy call site served by the B200 path.

CPU tier: the recogniser (expression graph -> the literals of api.solve) on models wired the way the reference scripts
wire them (arbitrage.py:38-78, liquidation.py:38-81, two-asset.py:40-87), the write-back of `.value`s with the ORACLE
installed as the checker back end, the error messages for models outside the routing family, and a cvxpy script of the
reference's kind (tests/routing_script.py), unmodified, through `run_script`.  GPU tier: the same models with the real
back end against the fixture of the executed reference (tests/golden/reference_run.json)."""
import json
import os
import types

import numpy as np
import pytest

import cfmm_routing_code_b200 as cf
import cfmm_routing_code_b200.cvxpy_compat as cp
from cfmm_routing_code_b200 import instances as I, run_script
from oracle import cfmm_oracle as O
import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref_run():
    with open(os.path.join(ROOT, "tests", "golden", "reference_run.json")) as f:
        return json.load(f)


def oracle_backend(local_indices, reserves, fees, kinds, weights, utility=None, n_tokens=None, tol=1e-9, verbose=False):
    """the oracle behind api.solve's signature (tests only)"""
    hp = cf.HostPools.from_lists(n_tokens, local_indices, reserves, fees, kinds, weights)
    sp = utility.spec(n_tokens)
    r = O.solve(H.oracle_pools(hp), O.Utility(sp.c, sp.a, sp.eq, sp.pinned), tol=tol)
    return types.SimpleNamespace(value=r.value, psi=r.psi, deltas=r.deltas, lambdas=r.lambdas, status=r.status)


@pytest.fixture
def with_oracle_backend(monkeypatch):
    monkeypatch.setattr(cp, "_backend", oracle_backend)


def pools_model(d):
    """trade variables, net flow psi and the trading-function constraints of a list-form problem, in cvxpy terms
    (what arbitrage.py:42-74 states for its five pools)"""
    n = d["n_tokens"]
    deltas = [cp.Variable(len(l), nonneg=True) for l in d["local_indices"]]
    lambdas = [cp.Variable(len(l), nonneg=True) for l in d["local_indices"]]
    psi = cp.sum([np.eye(n)[:, l] @ (L - D) for l, D, L in zip(d["local_indices"], deltas, lambdas)])
    cons = []
    for R, g, D, L, kind, w in zip(d["reserves"], d["fees"], deltas, lambdas, d["kinds"], d["weights"]):
        R = np.array(R, float)
        x = R + g * D - L
        if kind == "sum":
            cons += [cp.sum(x) >= cp.sum(R), x >= 0]
        elif kind == "bounded_product":              # INTEGRATION.md: product on virtual reserves R + o, real reserves >= 0
            cons += [cp.geo_mean(x + np.array(w)) >= cp.geo_mean(R + np.array(w)), x >= 0]
        else:
            p = None if kind == "product" else np.array(w)
            cons.append(cp.geo_mean(x, p=p) >= cp.geo_mean(R, p=p))
    return psi, deltas, lambdas, cons


def wire(d, objective, token_constraints):
    psi, deltas, lambdas, cons = pools_model(d)
    return cp.Problem(cp.Maximize(objective(psi)), cons + token_constraints(psi)), psi, deltas, lambdas


def arbitrage_model():
    d = I.arbitrage_instance()
    return d, wire(d, lambda psi: np.array(d["market_value"]) @ psi, lambda psi: [psi >= 0])


def liquidation_model():
    d = I.liquidation_instance()
    ca = d["current_assets"]
    return d, wire(d, lambda psi: psi[4], lambda psi: [psi[j] + ca[j] == 0 for j in range(4)])


def swap_model(t):
    d = I.two_asset_instance()
    assets = np.array([t, 0, 0])
    return d, wire(d, lambda psi: psi[2], lambda psi: [psi + assets >= 0])


def check_literals(m, d):
    assert m.n_tokens == d["n_tokens"] and m.local_indices == d["local_indices"] and m.kinds == d["kinds"]
    assert [list(map(float, r)) for r in m.reserves] == [list(map(float, r)) for r in d["reserves"]]
    assert m.fees == [float(f) for f in d["fees"]]
    w0 = np.asarray(d["weights"][0], float)
    assert np.array_equal(m.weights[0], w0 / w0.sum()) and all(w is None for w in m.weights[1:])


def test_recogniser_recovers_the_literals_of_the_three_scripts():
    d, (prob, *_) = arbitrage_model()
    m = cp.recognise(prob.objective, prob.constraints)
    check_literals(m, d)
    s = cf.Arbitrage(d["market_value"]).spec(4)
    assert np.array_equal(m.c, s.c) and np.array_equal(m.a, s.a) and not m.eq.any() and not m.pinned.any()
    d, (prob, *_) = liquidation_model()
    m = cp.recognise(prob.objective, prob.constraints)
    check_literals(m, d)
    s = cf.Liquidate(d["target"], d["current_assets"]).spec(5)
    assert np.array_equal(m.c, s.c) and np.array_equal(m.a, s.a) and np.array_equal(m.eq, s.eq) and np.array_equal(m.pinned, s.pinned)
    for t in (0.0, 12.5):
        d, (prob, *_) = swap_model(t)
        m = cp.recognise(prob.objective, prob.constraints)
        check_literals(m, d)
        s = cf.Swap(0, 2, t).spec(3)
        assert np.array_equal(m.c, s.c) and np.array_equal(m.a, s.a) and not m.eq.any() and not m.pinned.any()


def test_solve_writes_back_what_the_scripts_read(with_oracle_backend, ref_run):
    d, (prob, psi, deltas, lambdas) = arbitrage_model()
    g = ref_run["arbitrage"]
    assert psi.value is None and prob.value is None
    v = prob.solve(solver="ECOS", warm_start=True)      # cvxpy's back-end selectors are accepted and ignored
    assert prob.status == "optimal" and v == prob.value and abs(v - g["value"]) <= 1e-8 * abs(g["value"])      # arbitrage.py:84
    np.testing.assert_allclose(psi.value, g["psi"], atol=2e-6)
    for i in range(5):
        np.testing.assert_allclose(deltas[i].value, g["deltas"][i], atol=5e-5)
        np.testing.assert_allclose(lambdas[i].value, g["lambdas"][i], atol=5e-5)
    assert abs(prob.objective.value - v) == 0.0
    d, (prob, psi, deltas, lambdas) = liquidation_model()
    g = ref_run["liquidation"]
    prob.solve()
    assert prob.status == "optimal" and abs(psi.value[4] - g["value"]) <= 1e-8 * g["value"]                    # liquidation.py:87
    np.testing.assert_allclose(psi.value, g["psi"], atol=2e-6)
    g = ref_run["two_asset"]
    amounts = I.two_asset_instance()["amounts"]
    for j in (0, 7, 49):
        d, (prob, psi, deltas, lambdas) = swap_model(amounts[j])
        prob.solve()
        assert abs(prob.objective.value - g["u_t"][j]) <= 1e-7 * max(abs(g["u_t"][j]), 1.0)                    # two-asset.py:100
        for k in range(5):                                                                                       # two-asset.py:94
            np.testing.assert_allclose(lambdas[k].value - deltas[k].value, g["flows"][j][k], atol=5e-5)


def test_expression_algebra_matches_numpy():
    rng = np.random.default_rng(0)
    x, y = cp.Variable(3, nonneg=True), cp.Variable(2)
    M, v, w = rng.normal(size=(4, 3)), rng.normal(size=4), rng.normal(size=3)
    e = 2.0 * (M @ (x - w)) + v - (M @ x) / 4.0 + np.float64(0.5) * (M @ x)
    x.value, y.value = rng.normal(size=3), rng.normal(size=2)
    np.testing.assert_allclose(e.value, 2.0 * (M @ (x.value - w)) + v - (M @ x.value) / 4.0 + 0.5 * (M @ x.value), rtol=1e-14)
    assert e.shape == (4,) and e[1].shape == () and e[1:3].shape == (2,) and (v @ e).shape == () and len(e) == 4
    assert abs((v @ e).value - v @ e.value) <= 1e-12 and abs((e @ v).value - v @ e.value) <= 1e-12
    assert abs(cp.sum(e).value - e.value.sum()) <= 1e-12 and cp.sum(np.arange(4.0)) == 6.0
    np.testing.assert_allclose((w * x + y[0]).value, w * x.value + y.value[0], rtol=1e-14)
    np.testing.assert_allclose((1.0 - x).value, 1.0 - x.value, rtol=1e-14)
    np.testing.assert_allclose(cp.sum([x, x, w]).value, 2 * x.value + w, rtol=1e-14)
    assert cp.geo_mean(np.array([4.0, 4, 4, 4])) == pytest.approx(4.0)
    assert cp.geo_mean([2.0, 8.0], p=[3, 1]) == pytest.approx(2.0 ** 0.75 * 8.0 ** 0.25)
    c = (e >= 1.0)
    assert isinstance(c, cp.Constraint) and c.op == ">=" and np.allclose(c.expr.value, e.value - 1.0)
    c = (1.0 >= e[0])
    assert c.op == ">=" and abs(c.expr.value - (1.0 - e.value[0])) <= 1e-12
    assert (e[0] == 2.0).op == "=="
    assert len(cp.Problem(cp.Maximize(e[0]), [e >= 0, y >= 1]).variables()) == 2
    z = cp.Variable()                                   # scalar variable
    z.value = 3.0
    assert z.shape == () and z.value == 3.0 and (2 * z + 1).value == 7.0 and np.allclose((x + z).value, x.value + 3.0)


def test_models_outside_the_routing_family_are_refused_by_name():
    d = I.arbitrage_instance()

    def build(mutate):
        _, (prob, psi, deltas, lambdas) = arbitrage_model()
        return mutate(prob, psi, deltas, lambdas)

    def expect(msg, mutate):
        with pytest.raises(cp.NotRoutingProblem, match=msg):
            prob = build(mutate)
            cp.recognise(prob.objective, prob.constraints)

    def other_level(prob, psi, deltas, lambdas):        # phi(new) >= 1.01 phi(R): not the trading-function constraint
        R = np.array(d["reserves"][1], float)
        prob.constraints[1] = cp.geo_mean(R + 0.997 * deltas[1] - lambdas[1]) >= 1.01 * cp.geo_mean(R)
        return prob
    expect("differs from the trading function", other_level)

    def coupled(prob, psi, deltas, lambdas):
        prob.constraints.append(psi[0] + psi[1] >= 0)
        return prob
    expect("couples the net flows of several tokens", coupled)

    def gross(prob, psi, deltas, lambdas):              # a constraint on what is tendered alone, not on the net flow
        prob.constraints.append(1.0 - deltas[1][0] >= 0)
        return prob
    expect("net flow", gross)

    def no_positivity(prob, psi, deltas, lambdas):      # constant sum without new_reserves >= 0
        del prob.constraints[5]
        return prob
    expect("without new_reserves >= 0", no_positivity)

    def upper(prob, psi, deltas, lambdas):
        prob.constraints.append(5.0 - psi[2] >= 0)
        return prob
    expect("upper bound", upper)

    def unvalued(prob, psi, deltas, lambdas):           # objective drops token 0 and nothing constrains it
        prob.objective = cp.Maximize(psi[1])
        prob.constraints[-1] = psi[1:] >= 0
        return prob
    expect("neither the objective nor any constraint", unvalued)

    with pytest.raises(cp.NotRoutingProblem, match="nonneg=True"):
        R = np.array([10.0, 1.0])
        D, L = cp.Variable(2), cp.Variable(2, nonneg=True)
        cp.recognise(cp.Maximize((L - D)[0] + (L - D)[1]), [cp.geo_mean(R + 0.997 * D - L) >= cp.geo_mean(R), L - D >= 0])
    with pytest.raises(cp.NotRoutingProblem, match="both contain variables"):
        x = cp.Variable(2)
        x * x
    with pytest.raises(cp.NotRoutingProblem, match="Maximize"):
        cp.Problem(cp.Variable(2)[0], [])


def test_minimize_and_equal_weight_geomean_and_infeasible(with_oracle_backend):
    # one 3-token equal-weight pool + two product pools; Minimize(-value) is the same program as Maximize(value)
    R3, Ra, Rb = np.array([30.0, 20.0, 10.0]), np.array([10.0, 8.0]), np.array([5.0, 9.0])
    A = [np.eye(3), np.eye(3)[:, [0, 1]], np.eye(3)[:, [1, 2]]]
    out = []
    for sense in (cp.Maximize, cp.Minimize):
        D = [cp.Variable(k, nonneg=True) for k in (3, 2, 2)]
        L = [cp.Variable(k, nonneg=True) for k in (3, 2, 2)]
        psi = cp.sum([A_i @ (l - d) for A_i, d, l in zip(A, D, L)])
        val = np.array([1.0, 2.0, 5.0]) @ psi
        cons = [cp.geo_mean(R + 0.997 * d - l) >= cp.geo_mean(R) for R, d, l in zip((R3, Ra, Rb), D, L)] + [psi >= 0]
        prob = cp.Problem(sense(val if sense is cp.Maximize else -val), cons)
        prob.solve()
        assert prob.model.kinds == ["geomean", "product", "product"] and np.allclose(prob.model.weights[0], 1 / 3)
        out.append((prob.value, psi.value))
    assert out[0][0] > 0 and abs(out[0][0] + out[1][0]) <= 1e-9 * out[0][0]
    np.testing.assert_allclose(out[0][1], out[1][1], atol=1e-7)


def wire_general(d, util):
    """any list-form problem and any linear + box utility"""
    psi, deltas, lambdas, cons = pools_model(d)
    for j in range(d["n_tokens"]):
        if not util.pinned[j]:
            cons.append(psi[j] + util.a[j] == 0 if util.eq[j] else psi[j] + util.a[j] >= 0)
    return cp.Problem(cp.Maximize(util.c @ psi), cons), psi, deltas, lambdas


def test_random_models_round_trip(with_oracle_backend):
    """random problems of the reference's scale, every pool kind and utility: the recogniser returns the literals the model
    was wired from, and prob.solve() leaves the oracle's optimum in the script-side expressions"""
    rng = np.random.default_rng(11)
    done = 0
    for _ in range(12):
        hp, d, prices = H.random_small_problem(rng, all_kinds=True)
        for util in H.random_utilities(rng, d["n_tokens"], prices):
            prob, psi, deltas, lambdas = wire_general(d, util)
            m = cp.recognise(prob.objective, prob.constraints)
            assert m.local_indices == d["local_indices"] and m.kinds == d["kinds"] and m.fees == d["fees"]
            assert all(np.allclose(r, r0, rtol=1e-15, atol=0) for r, r0 in zip(m.reserves, d["reserves"]))
            for w, w0, kind in zip(m.weights, d["weights"], d["kinds"]):
                assert (w is None) == (w0 is None)
                if kind == "bounded_product":        # offsets come back as (R + o) - R
                    assert np.allclose(w, w0, rtol=1e-12)
                elif w is not None:
                    assert np.allclose(w, np.asarray(w0) / np.sum(w0), rtol=1e-15)
            assert np.array_equal(m.c, util.c) and np.array_equal(m.eq, util.eq) and np.array_equal(m.pinned, util.pinned)
            assert np.array_equal(m.a, np.where(util.pinned, 0.0, util.a))
            ro = O.solve(H.oracle_pools(hp), util, tol=1e-9)
            if ro.status != "optimal":
                continue
            prob.solve()
            assert prob.status == "optimal" and abs(prob.value - ro.value) <= 1e-8 * max(abs(ro.value), 1.0)
            np.testing.assert_allclose(psi.value, ro.psi, atol=1e-7 * max(np.abs(ro.psi).max(), 1.0))
            done += 1
    assert done >= 30


def test_cvxpy_script_runs_unmodified_through_the_compat_module(with_oracle_backend, ref_run, capsys):
    """tests/routing_script.py states the three problems of the reference's scripts with `import cvxpy as cp` and plots
    with matplotlib; run_script serves both, and what the script reads back is the executed reference's"""
    g = run_script.run(os.path.join(ROOT, "tests", "routing_script.py"))
    assert abs(g["prob"].value - ref_run["arbitrage"]["value"]) <= 1e-8 * ref_run["arbitrage"]["value"]
    assert g["prob"].model.local_indices == ref_run["arbitrage"]["data"]["local_indices"]
    assert abs(g["liq_psi"].value[4] - ref_run["liquidation"]["value"]) <= 1e-8 * ref_run["liquidation"]["value"]
    out = capsys.readouterr().out
    assert "Total output value: 21.4998" in out and "Total liquidated value: 15.8830" in out
    np.testing.assert_allclose(g["u_t"], ref_run["two_asset"]["u_t"], rtol=1e-7, atol=1e-7)
    for k in range(5):                                                      # fixture: [t][pool][slot]; two-asset.py:93-94
        np.testing.assert_allclose(g["all_values"][k], np.array([flows_t[k] for flows_t in ref_run["two_asset"]["flows"]]).T, atol=5e-5)


@pytest.mark.gpu
def test_cuda_back_end_serves_the_cvxpy_call_site(ref_run):
    """prob.solve() of the scripts' models = api.solve on the GPU; what the scripts read back vs the executed reference"""
    assert cp._backend is None
    d, (prob, psi, deltas, lambdas) = arbitrage_model()
    g = ref_run["arbitrage"]
    prob.solve()
    assert prob.status == "optimal" and abs(prob.value - g["value"]) <= 1e-8 * abs(g["value"])
    np.testing.assert_allclose(psi.value, g["psi"], atol=1e-6 * np.abs(g["psi"]).max())
    for i in range(5):
        np.testing.assert_allclose(deltas[i].value, g["deltas"][i], atol=5e-5)
        np.testing.assert_allclose(lambdas[i].value, g["lambdas"][i], atol=5e-5)
    d, (prob, psi, deltas, lambdas) = liquidation_model()
    g = ref_run["liquidation"]
    prob.solve()
    assert prob.status == "optimal" and abs(psi.value[4] - g["value"]) <= 1e-8 * g["value"]
    g = ref_run["two_asset"]
    amounts = I.two_asset_instance()["amounts"]
    for j in range(0, 50, 7):
        d, (prob, psi, deltas, lambdas) = swap_model(amounts[j])
        prob.solve()
        assert prob.status == "optimal" and abs(prob.objective.value - g["u_t"][j]) <= 1e-7 * max(abs(g["u_t"][j]), 1.0)
        for k in range(5):
            np.testing.assert_allclose(lambdas[k].value - deltas[k].value, g["flows"][j][k], atol=5e-5)
