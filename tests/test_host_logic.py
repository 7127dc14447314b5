"""Host-side logic of the product, on CPU: solver.py driven by the oracle-backed evaluator, pool bucketing
and sharding, the C ABI's symbol table, loud failure without a GPU, and the world_size=2 all-reduce path (gloo)."""
import ctypes
import os
import re
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import cfmm_routing_code_b200 as cf
from oracle import cfmm_oracle as O
from cfmm_routing_code_b200 import _lib, instances as I, pools as PL
from cfmm_routing_code_b200.solver import Comm, solve_dual
from cpu_evaluator import OracleEvaluator
import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    text = ""
    for fn in sorted(os.listdir(os.path.join(ROOT, "include"))):
        if fn.endswith(".h"):
            text += open(os.path.join(ROOT, "include", fn)).read()
    names = set(re.findall(r"\b(cfmm_[a-z0-9_]+)\s*\(", text))
    assert len(names) >= 12
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/ but not exported by libcfmm_b200.so"
    assert b"sm_100a" in lib.cfmm_version()
    # argument validation happens before any CUDA call, so it is testable without a GPU
    b = _lib.Bucket(_lib.KIND_PRODUCT, 2, 10, 10, None, None, None, None, None, None)
    assert lib.cfmm_arb_eval(ctypes.byref(b), 4, None, None, 0.0, None, None, None, None) == -1
    b = _lib.Bucket(9, 2, 0, 0, 1, 1, 1, None, None, None)
    assert lib.cfmm_arb_eval(ctypes.byref(b), 4, None, None, 0.0, None, None, None, None) == -2
    assert lib.cfmm_blocked_eval(None, 4, None, None, None, None, None, 0, None) == -1
    # batch entry points: NULL / size / kind checks, work-buffer arithmetic (12 n + 2 n^2 + n(n+1) + 2 nnz doubles per lane)
    assert lib.cfmm_batch_solve(None, None, None, None, None) == -1
    cp = _lib.CsrPools(3, 5, 13, None, None, None, None, None, None, None)
    assert lib.cfmm_set_batch_lanes(1) == 0         # the lane count is process-wide: a batch solve run earlier sets it
    assert lib.cfmm_batch_solve_work_bytes(ctypes.byref(cp), 50, 0) == 8 * (36 + 18 + 12 + 26) * 64
    assert lib.cfmm_batch_solve_work_bytes(ctypes.byref(cp), 50, 6) == 8 * (36 + 18 + 12 + 12) * 64
    assert lib.cfmm_set_batch_lanes(5) == -2 and lib.cfmm_set_batch_lanes(32) == 0
    assert lib.cfmm_batch_solve_work_bytes(ctypes.byref(cp), 50, 0) == 8 * (36 + 18 + 12 + 26) * 64 * 32
    assert lib.cfmm_set_batch_lanes(1) == 0
    big = _lib.CsrPools(65, 5, 13, None, None, None, None, None, None, None)
    assert lib.cfmm_batch_solve_work_bytes(ctypes.byref(big), 50, 0) == -3
    bt = _lib.Batch(1, None, None, None, None, None, None, None, None, None, 0)
    prm = _lib.BatchParams(1e-8, 0.1, 1e-4, 0.25, 1e-12, 60, 100)
    assert lib.cfmm_batch_solve(ctypes.byref(cp), ctypes.byref(bt), ctypes.byref(prm), None, None) == -1


def test_native_solver_work_buffer_covers_the_hcoef_slab():
    """cfmm_blocked_solve carves an hcoef slab of the layout's slab stride (n_tiles * P) from the caller's work buffer"""
    lib = _lib.load()
    n = 4096
    for m, tiles in ((1_000_000, 1117), (1001, 2)):
        b = _lib.BlockedPairs(m, tiles, 896, 0, None, None, None, None, None, None, None, None)
        need = lib.cfmm_blocked_solve_work_bytes(ctypes.byref(b), n)
        assert need >= 8 * tiles * 896 + 8 * (2 * (n + 1) + 15 * n), (m, tiles, need)


def test_product_path_fails_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    d = I.arbitrage_instance()
    with pytest.raises(cf.CfmmError):
        cf.solve(d["local_indices"], d["reserves"], d["fees"], d["kinds"], d["weights"],
                 utility=cf.Arbitrage(d["market_value"]))
    with pytest.raises(cf.CfmmError):
        cf.PoolStore(H.host_pools(d), device="cpu")


@pytest.mark.parametrize("linear_solver", ["dense", "cg"])
def test_solver_logic_reproduces_the_reference_instances(golden, linear_solver):
    d = I.arbitrage_instance()
    r = solve_dual(OracleEvaluator(H.host_pools(d)), cf.Arbitrage(d["market_value"]).spec(4), tol=1e-9,
                   linear_solver=linear_solver)
    assert r.status == "optimal" and abs(r.primal_value - golden["arbitrage"]["value"]) <= 1e-7
    np.testing.assert_allclose(r.psi.numpy(), golden["arbitrage"]["psi"], atol=2e-6)
    d = I.liquidation_instance()
    r = solve_dual(OracleEvaluator(H.host_pools(d)), cf.Liquidate(4, d["current_assets"]).spec(5), tol=1e-9,
                   linear_solver=linear_solver)
    assert r.status == "optimal" and abs(r.primal_value - golden["liquidation"]["value"]) <= 1e-7
    d = I.two_asset_instance()
    hp = H.host_pools(d)
    for j in (0, 10, 20, 35, 49):
        r = solve_dual(OracleEvaluator(hp), cf.Swap(0, 2, d["amounts"][j]).spec(3), tol=1e-9,
                       linear_solver=linear_solver)
        assert abs(r.primal_value - golden["two_asset"][j]["value"]) <= 2e-7 * max(1, golden["two_asset"][j]["value"])


def test_solver_logic_on_synthetic_mixed_pools_certifies_its_answer():
    hp, s = H.mixed_host_pools(3000, 60, seed=4)
    r = solve_dual(OracleEvaluator(hp), cf.Arbitrage(s["prices"]).spec(60), tol=1e-8)
    assert r.status == "optimal" and abs(r.gap) <= 1e-7 and r.primal_infeas <= 1e-7


# ---- CPU twins of the solve-level GPU parity tests (tests/test_gpu_parity.py): same instances, same assertions, the
# product's outer loop over the CPU stand-in evaluator -- a regression in the outer loop shows up here, without a GPU
def test_cpu_twin_cfg2_solve_matches_oracle():
    hp, s = H.cp_host_pools(10_000, 256, seed=0)
    for ls in ("cg", "dense"):
        r = solve_dual(OracleEvaluator(hp), cf.Arbitrage(s["prices"]).spec(256), tol=1e-9, linear_solver=ls)
        ro = O.solve(H.oracle_pools(hp), O.Utility.arbitrage(s["prices"]), tol=1e-10)
        assert r.status == "optimal" and ro.status == "optimal"
        assert abs(r.primal_value - ro.value) <= 1e-8 * abs(ro.value)
        assert abs(r.gap) <= 1e-8 and r.primal_infeas <= 1e-8
        gross = np.zeros(256); np.add.at(gross, hp.tok_idx, np.concatenate(ro.deltas) + np.concatenate(ro.lambdas))
        assert np.max(np.abs(r.psi.numpy() - ro.psi) / gross.max()) <= 1e-7


def test_cpu_twin_cfg3_small_mixed_solve_matches_oracle():
    hp, s = H.mixed_host_pools(8000, 150, seed=1)
    r = solve_dual(OracleEvaluator(hp), cf.Arbitrage(s["prices"]).spec(150), tol=1e-8)
    ro = O.solve(H.oracle_pools(hp), O.Utility.arbitrage(s["prices"]), tol=1e-9)
    assert r.status == "optimal"
    assert abs(r.primal_value - ro.value) <= 1e-6 * abs(ro.value)
    assert abs(r.gap) <= 1e-6 and r.primal_infeas <= 1e-6
    # per-token complementarity (arbitrage.py:77): psi >= 0 to 1e-6 of the largest flow
    assert r.psi.numpy().min() >= -1e-6 * np.abs(ro.psi).max()


def test_cpu_twin_cfg4_small_liquidation_matches_oracle():
    """the case that failed on the B200 in round 1: 'optimal' at tol 1e-8 with one cheap token's equality off by 6.3e-5"""
    hp, s = H.mixed_host_pools(8000, 150, seed=2)
    basket = I.synth_basket(150, s["prices"], seed=2)
    nu0 = s["prices"] / s["prices"][0]
    r = solve_dual(OracleEvaluator(hp), cf.Liquidate(0, basket).spec(150), nu0=nu0, tol=1e-8)
    ro = O.solve(H.oracle_pools(hp), O.Utility.liquidate(150, 0, basket), nu0=nu0, tol=1e-9)
    assert r.status == "optimal"
    assert abs(r.primal_value - ro.value) <= 1e-6 * abs(ro.value)
    # liquidation.py:77-80: psi_j + a_j == 0 token by token, to 1e-6 of the basket scale (in fact to ~tol)
    np.testing.assert_allclose(r.psi.numpy()[1:], -basket[1:], atol=1e-6 * basket.max())
    np.testing.assert_allclose(ro.psi[1:], -basket[1:], atol=1e-6 * basket.max())
    assert np.abs(r.psi.numpy()[1:] + basket[1:]).max() <= 1e-7 * basket.max()


def test_infeasible_problems_are_flagged_not_reported_optimal():
    """cvxpy's prob.status == 'infeasible' (arbitrage.py:82): a token that must be RECEIVED in a quantity the pools cannot
    deliver -- the dual is unbounded (its price runs away) and the solve ends uncertified; api.infeasible_suspected turns
    that pattern into status 'infeasible'.  A feasible problem that merely ran out of iterations keeps 'max_iter'."""
    from cfmm_routing_code_b200.api import infeasible_suspected
    hp = cf.HostPools.from_lists(2, [[0, 1]], [[10.0, 10.0]], [0.997], ["product"], [None])
    spec = cf.DualSpec(np.array([1.0, 0.0]), np.array([0.0, -100.0]), np.array([False, True]), np.array([True, False]))
    r = solve_dual(OracleEvaluator(hp), spec, tol=1e-8, max_inner=60)
    assert r.status != "optimal"
    assert infeasible_suspected(spec, r.nu.numpy(), r.psi.numpy(), r.status)
    # the same pool can deliver 5 units: feasible, certified, not flagged
    spec2 = cf.DualSpec(np.array([1.0, 0.0]), np.array([0.0, -5.0]), np.array([False, True]), np.array([True, False]))
    r2 = solve_dual(OracleEvaluator(hp), spec2, tol=1e-8)
    assert r2.status == "optimal" and not infeasible_suspected(spec2, r2.nu.numpy(), r2.psi.numpy(), r2.status)
    assert abs(float(r2.psi[1]) - 5.0) <= 1e-7
    # a feasible problem stopped early is 'max_iter', not 'infeasible'
    hp3, s3 = H.cp_host_pools(2000, 40, seed=3)
    sp3 = cf.Arbitrage(s3["prices"]).spec(40)
    r3 = solve_dual(OracleEvaluator(hp3), sp3, tol=1e-12, max_inner=2)
    assert r3.status == "max_iter" and not infeasible_suspected(sp3, r3.nu.numpy(), r3.psi.numpy(), r3.status)


def test_solver_logic_on_random_small_problems_matches_the_oracle():
    """the product's python outer loop (dense Newton path, look-ahead on) on 45 random problems of the reference's
    scale, evaluations by the CPU stand-in for PoolStore: same optimal values as the oracle's own solve"""
    rng = np.random.default_rng(21)
    for _ in range(15):
        hp, d, prices = H.random_small_problem(rng)
        op = H.oracle_pools(hp)
        for u in H.random_utilities(rng, hp.n_tokens, prices):
            r = solve_dual(OracleEvaluator(hp), cf.DualSpec(u.c, u.a, u.eq, u.pinned), tol=1e-8)
            ro = O.solve(op, u, tol=1e-8)
            assert abs(r.primal_value - ro.value) <= 1e-7 * max(abs(ro.dual_value), 1e-300)
            assert abs(r.gap) <= 1e-7 and r.primal_infeas <= 1e-7


def test_utilities_and_input_validation():
    assert cf.Liquidate(4, [2, 1, 3, 5, 10]).spec(5).pinned.tolist() == [False] * 4 + [True]
    sp = cf.Swap(0, 2, 7.5).spec(3)
    assert sp.a.tolist() == [7.5, 0, 0] and sp.c.tolist() == [0, 0, 1]
    with pytest.raises(ValueError):
        cf.Arbitrage([1.0, -2.0])
    with pytest.raises(ValueError):
        cf.HostPools.from_lists(3, [[0, 1, 2]], [[1, 1, 1]], [0.99], ["sum"])
    with pytest.raises(ValueError):
        cf.HostPools.from_lists(3, [[0, 0]], [[1, 1]], [0.99], ["product"])
    with pytest.raises(ValueError):
        cf.HostPools.from_lists(3, [[0, 1]], [[1, 1, 1]], [0.99], ["product"])
    with pytest.raises(ValueError):
        cf.HostPools.from_pairs(2, [[0, 1]], [[1.0, -1.0]], [0.99]).validate()
    with pytest.raises(ValueError):
        cf.HostPools.from_pairs(2, [[0, 5]], [[1.0, 1.0]], [0.99]).validate()
    with pytest.raises(ValueError):
        cf.solve([[0, 1]], [[1, 1]], [0.99], ["product"])          # utility is required


def test_bucketing_and_pool_sharding_partition_the_problem():
    hp, _ = H.mixed_host_pools(5000, 80, seed=9)
    whole = PL.split_buckets(hp)
    assert sum(b.m for b in whole) == hp.m
    kinds = {(b.kind, b.arity) for b in whole}
    assert (_lib.KIND_PRODUCT, 2) in kinds and (_lib.KIND_SUM, 2) in kinds and (_lib.KIND_GEOMEAN, 5) in kinds
    for world in (2, 3, 8):
        seen = []
        for rank in range(world):
            seen += [b.sel for b in PL.split_buckets(hp, rank, world)]
        allsel = np.sort(np.concatenate(seen))
        assert np.array_equal(allsel, np.arange(hp.m))          # every pool on exactly one rank
    # constant-product-only problems take the no-gather fast path
    hp2, _ = H.cp_host_pools(1000, 16, seed=1)
    (b,) = PL.split_buckets(hp2)
    assert b.identity and b.kind == _lib.KIND_PRODUCT and np.array_equal(b.off[:, 3], [6, 7])


def test_bounded_product_pools_get_their_own_bucket():
    d = I.v3_instance(); hp = H.host_pools(d)
    hp.validate()
    specs = PL.split_buckets(hp)
    by_kind = {(b.kind, b.arity): b for b in specs}
    assert set(by_kind) == {(_lib.KIND_BOUNDED, 2), (_lib.KIND_PRODUCT, 2), (_lib.KIND_GEOMEAN, 3)}
    b = by_kind[(_lib.KIND_BOUNDED, 2)]
    assert b.sel.tolist() == [0, 1, 2] and np.array_equal(hp.weights[b.off], np.array(d["weights"][:3]).T)
    assert hp.reserves[hp.pool_ptr[1] + 1] == 0.0            # the out-of-range position holds token 0 only
    db = PL.DeviceBucket(hp, b, "cpu")                        # slot-major SoA the kernel reads (tensors only, no launch)
    assert db.kind == _lib.KIND_BOUNDED and db.stride == 1024 and db.theta_bar is None and db.logrw is None
    np.testing.assert_array_equal(db.weights[:, :3].numpy(), np.array(d["weights"][:3]).T)      # offsets ride in weights
    np.testing.assert_array_equal(db.reserves[:, :3].numpy(), np.array(d["reserves"][:3]).T)
    np.testing.assert_array_equal(db.tok_idx[:, :3].numpy(), np.array(d["local_indices"][:3]).T)
    assert db.c_bucket.kind == 3 and db.c_bucket.arity == 2 and db.c_bucket.n_pools == 3 and db.c_bucket.weights
    with pytest.raises(ValueError):
        cf.HostPools.from_lists(3, [[0, 1, 2]], [[1, 1, 1]], [0.99], ["bounded_product"], [[1, 1, 1]])
    with pytest.raises(ValueError):
        cf.HostPools.from_lists(2, [[0, 1]], [[0.0, 1.0]], [0.99], ["bounded_product"], [[0.0, 1.0]]).validate()


def test_blocked_layout_builder_tables_reproduce_the_scatter():
    """build_blocked_pairs on CPU tensors: emulate the kernel's row sums (cfmm_blocked.cuh: pool phase scatters the flows
    into row order, one thread sums each row) and compare with index_add"""
    lib = _lib.load()
    assert lib.cfmm_set_blocked_config(400 + 1024) == -2               # tile size is a compile-time constant now
    P, rs, ts, cap = PL.blocked_layout_info(lib)
    assert P == 896 and rs == P + P // 4 + 8 and ts == P and cap == 32
    for m, n in ((5000, 300), (700, 3), (40_000, 2000), (9_000, 50)):
        s = I.synth_const_product(m, n, 0)
        idx = torch.as_tensor(s["idx"].T.astype(np.int64).copy())
        order, res, t = PL.build_blocked_pairs(idx, n, P, rs, ts, cap)
        assert len(order) + len(res) == m and t is not None
        H.check_blocked_tables(t, idx, order, n, P, rs, ts, cap)


# ---------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_main(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        hp, s = H.mixed_host_pools(2000, 40, seed=6)
        comm = Comm()
        assert comm.dist is not None
        r = solve_dual(OracleEvaluator(hp, rank, world), cf.Arbitrage(s["prices"]).spec(40), tol=1e-9, comm=comm)
        q.put((rank, r.primal_value, r.psi.numpy(), r.nu.numpy(), r.status, comm.calls, r.evals))
    finally:
        dist.destroy_process_group()


def test_pool_sharded_solve_over_gloo_world2_matches_single_process():
    """SURVEY 8e: pools shard across ranks, nu is replicated, ONE all-reduce of [psi | arb] per evaluation."""
    hp, s = H.mixed_host_pools(2000, 40, seed=6)
    single = solve_dual(OracleEvaluator(hp), cf.Arbitrage(s["prices"]).spec(40), tol=1e-9)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted([q.get(timeout=240) for _ in procs], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, val, psi, nu, status, calls, evals in outs:
        assert status == "optimal"
        assert abs(val - single.primal_value) <= 1e-8 * abs(single.primal_value)
        assert calls >= evals                      # at least one all-reduce per dual evaluation
    # every rank applied the same update: prices are bit-identical across ranks
    assert np.array_equal(outs[0][3], outs[1][3])
    np.testing.assert_allclose(outs[0][2], single.psi.numpy(), atol=1e-7 * np.abs(single.psi.numpy()).max())
