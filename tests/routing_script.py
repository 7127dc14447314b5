"""A cvxpy script of the kind the reference ships: its three routing problems (cfmm_routing_code_b200.instances) stated
with cvxpy's modelling API, solved by prob.solve(), read back from .value, printed, and the swap sweep plotted.

Not a test module.  tests/test_cvxpy_compat.py runs it through cfmm_routing_code_b200.run_script (`import cvxpy` is the
compat module) and tests/test_reference_pin.py with oracle/cvxpy_shim.py standing in for cvxpy; both compare the globals
it leaves with what the reference's own scripts produced (tests/golden/reference_run.json)."""
import cvxpy as cp
import matplotlib.pyplot as plt
import numpy as np

from cfmm_routing_code_b200 import instances as I


def routing_problem(d, objective, token_constraints):
    """trade variables, net flow psi and the trading-function constraints of a list-form problem"""
    n = d["n_tokens"]
    deltas = [cp.Variable(len(l), nonneg=True) for l in d["local_indices"]]
    lambdas = [cp.Variable(len(l), nonneg=True) for l in d["local_indices"]]
    psi = cp.sum([np.eye(n)[:, l] @ (L - D) for l, D, L in zip(d["local_indices"], deltas, lambdas)])
    cons = []
    for R, g, D, L, kind, w in zip(d["reserves"], d["fees"], deltas, lambdas, d["kinds"], d["weights"]):
        R = np.array(R, float)
        new_reserves = R + g * D - L
        if kind == "sum":
            cons += [cp.sum(new_reserves) >= cp.sum(R), new_reserves >= 0]
        else:
            p = None if kind == "product" else np.array(w)
            cons.append(cp.geo_mean(new_reserves, p=p) >= cp.geo_mean(R, p=p))
    obj = objective(psi)
    return cp.Problem(cp.Maximize(obj), cons + token_constraints(psi)), obj, psi, deltas, lambdas


d = I.arbitrage_instance()
prob, _, psi, deltas, lambdas = routing_problem(d, lambda psi: np.array(d["market_value"]) @ psi, lambda psi: [psi >= 0])
prob.solve()
print(f"Total output value: {prob.value}")

d = I.liquidation_instance()
ca, target = d["current_assets"], d["target"]
liq_prob, _, liq_psi, liq_deltas, liq_lambdas = routing_problem(
    d, lambda psi: psi[target], lambda psi: [psi[j] + ca[j] == 0 for j in range(d["n_tokens"]) if j != target])
liq_prob.solve()
print(f"Total liquidated value: {liq_psi.value[target]}")

d = I.two_asset_instance()
amounts = d["amounts"]
u_t = np.zeros(len(amounts))
all_values = [np.zeros((len(l), len(amounts))) for l in d["local_indices"]]      # [pool][slot, t]: lambda - delta
for j, t in enumerate(amounts):
    tendered = np.zeros(d["n_tokens"])
    tendered[d["tok_in"]] = t
    swap, obj, _, sw_deltas, sw_lambdas = routing_problem(d, lambda psi: psi[d["tok_out"]], lambda psi: [psi + tendered >= 0])
    swap.solve()
    u_t[j] = obj.value
    for k, (D, L) in enumerate(zip(sw_deltas, sw_lambdas)):
        all_values[k][:, j] = L.value - D.value
print(f"Swap of {amounts[-1]} of token {d['tok_in']}: {u_t[-1]} of token {d['tok_out']}")

plt.figure()
plt.plot(amounts, u_t)
plt.xlabel("amount tendered")
plt.ylabel("amount received")
plt.show()
