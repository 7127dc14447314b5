#!/usr/bin/env python
"""bench.py -- pools x dual-evaluations / second on BASELINE.json configs[4] (1M constant-product pools, 4096 tokens,
pool-sharded over the N GPUs), plus wall-clock to 1e-6 relative gap, the HBM roofline of the dominant kernel, and the
CPU baseline timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--scaling strong|weak] [--dump-outputs DIR]

A "step" is one dual evaluation of the problem: the per-pool optimal-arbitrage kernel over this rank's pools,
accumulating psi(nu) and the dual value, + (N > 1) the one all-reduce of the (n_tokens+1)-vector.  Default scaling is
STRONG: the 1M pools are split over the N GPUs (BASELINE.json configs[4]); the weak-scaled figure (1M pools per GPU)
rides along as the `weak` key at N > 1.  Steps rotate over independent pool instances resident on each GPU, enough of
them to exceed the 126 MB L2 (>= 256 MiB), so every step streams its pools from HBM.  Exactly K steps are timed, replayed
from CUDA graphs.  One JSON line on stdout (rank 0).  --dump-outputs DIR writes what the last timed step returned, psi(nu)
as DIR/psi.npy and the dual value's arbitrage term as DIR/arb.npy (float64); the inputs are seeded, so two builds run with
the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

M_POOLS = 1_000_000
N_TOKENS = 4096
N_INSTANCES = 8
METRIC = "pools x dual-evaluations / second (1M constant-product pools, 4096 tokens); time to 1e-6 rel-gap reported beside it"
UNIT = "pool-evals/s"
E2E_REPS = 9             # repetitions of the end-to-end solve; the median is reported (host jitter on shared boxes: see profiles/r2z4_*)


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML; nvidia-smi as a fallback)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.sm, self.reasons, self.sm_max = [], set(), None
        self.stop = threading.Event()
        self.index = index
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None
        self.th = threading.Thread(target=self._run, daemon=True)

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40),
                          ("sw_thermal_slowdown", 0x20)):
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                              "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
        r = [x.strip() for x in out.strip().split(",")]
        if len(r) >= 6:
            self.sm.append(float(r[0])); self.sm_max = float(r[1])
            for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if r[2 + i] == "Active":
                    self.reasons.add(name)

    def _run(self):
        while not self.stop.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self.stop.wait(0.02)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml" if self.nvml else "nvidia-smi"}


# --------------------------------------------------------------------------------------------------
# CPU legs (the ONLY places this file executes oracle/)
# --------------------------------------------------------------------------------------------------
def _cfg5_host():
    from cfmm_routing_code_b200 import instances as I
    s = I.synth_const_product(M_POOLS, N_TOKENS, seed=3)
    return np.ascontiguousarray(s["idx"], np.int32), np.ascontiguousarray(s["reserves"]), s["gamma"], s["prices"]


def cpu_eval_throughput(seconds_budget=12.0, data=None):
    """oracle dual evaluations of the full 1M-pool instance on ALL host cores (oracle/cfmm_oracle_c.c, persistent
    pthread pool): pool-evals/s, number of evaluations, seconds, threads."""
    from oracle import c_oracle as CO
    idx, R, g, prices = data or _cfg5_host()
    nu = prices * np.exp(0.01 * np.random.default_rng(0).standard_normal(N_TOKENS))
    CO.autotune_threads(idx, R, g, N_TOKENS, nu)      # best thread count for this host (also warms up)
    t0 = time.perf_counter(); k = 0
    while True:
        CO.eval_pairs(idx, R, g, N_TOKENS, nu * (1 + 1e-3 * k)); k += 1
        dt = time.perf_counter() - t0
        if dt > seconds_budget or k >= 2000:
            break
    return M_POOLS * k / dt, k, dt, CO.num_threads()


def cpu_full_solve(data=None):
    """the whole solve to a 1e-6 certificate on the host cores: oracle_solve_pairs (C: projected Newton-PCG over the
    persistent pthread pool; oracle/cfmm_oracle_c.c) -- no product code on this path"""
    from oracle import c_oracle as CO
    idx, R, g, prices = data or _cfg5_host()
    CO.autotune_threads(idx, R, g, N_TOKENS, prices.copy())
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        nu, psi, res = CO.solve_pairs(idx, R, g, N_TOKENS, prices, tol=1e-6)
        wall = time.perf_counter() - t0
        if best is None or wall < best[0]:
            best = (wall, res)
    wall, res = best
    return {"value": M_POOLS * res.evals / wall, "unit": UNIT, "wall_s": wall, "evals": int(res.evals), "hvps": int(res.hvps),
            "status": {0: "optimal", 1: "max_iter", 2: "stalled"}[int(res.status)], "gap": float(res.gap),
            "threads": CO.num_threads()}


def run_reference(args):
    """The reference's path on the host cores.  cvxpy (the reference's solver) is probed at run time; it is not in this
    image, so the oracle port (oracle/cfmm_oracle_c.c: same dual evaluation and the same Newton-PCG outer loop, C +
    pthreads on all host cores) stands in -- kind 'port'.  The CPU has no shards: every N times the whole 1M-pool problem."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        import cvxpy  # noqa: F401
        have_cvxpy = True
    except Exception:
        have_cvxpy = False
    data = _cfg5_host()
    vals = []
    per_step_budget = max(1.0, min(15.0, 90.0 / max(args.steps + args.warmup, 1)))
    cores = 1
    for i in range(args.warmup + args.steps):
        v, k, dt, cores = cpu_eval_throughput(per_step_budget, data)
        if i >= args.warmup:
            vals.append((v, k, dt))
    value = float(np.mean([v for v, _, _ in vals]))
    sample = (f"{vals[0][1]} oracle dual evaluations of the full 1M-pool/4096-token instance per step "
              f"(C restatement oracle/cfmm_oracle_c.c, {cores} pthreads in a persistent pool, fp64)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean([dt / k for _, k, dt in vals])),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args.gpus, args.scaling, None),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "reference solver (cvxpy) " + ("present but not used for this metric" if have_cvxpy
                                                               else "unavailable in image")},
        "gpu_launches": 0,
    }
    solve = cpu_full_solve(data)
    line["e2e"] = {"value": solve["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "what": "one full solve to a 1e-6 certificate on the host cores (oracle_solve_pairs: the oracle's C "
                           "restatement of the dual Newton-PCG loop, no product code); value = pools x dual evaluations / wall",
                   "wall_s": solve["wall_s"], "evals": solve["evals"], "hvps": solve["hvps"], "status": solve["status"]}
    line["time_to_1e-6_gap"] = {"seconds": solve["wall_s"], "rel_gap": abs(solve["gap"]), "tol": 1e-6}
    print(json.dumps(line), flush=True)


def n_instances(per):
    """rotating pool instances per GPU: a multiple of 8 whose resident slabs exceed 256 MiB (> 2x the 126 MB L2)"""
    return 8 * max(1, -(-(256 << 20) // (8 * per * 32)))


def workload_config(n_gpus, scaling, n_inst):
    per = M_POOLS if scaling == "weak" else M_POOLS // n_gpus
    cfg = {"workload": f"BASELINE.json configs[4]: {per * n_gpus} constant-product pools in total "
                       f"({per} per GPU x {n_gpus}), 4096 tokens, Arbitrage(c=p), seeds 3+100k",
           "pools_total": per * n_gpus, "pools_per_gpu": per, "n_tokens": N_TOKENS, "parallelism": f"pool-shard x{n_gpus}",
           "collective": "none" if n_gpus == 1 else "one all-reduce of n_tokens+1 f64 per step"}
    if n_inst:
        cfg["l2"] = f"rotating {n_inst} pool instances per GPU ({n_inst * per * 32 // 2**20} MiB of slabs) > 126 MB L2"
    else:               # the CPU arm: the whole problem on the host cores, no shards, no L2 rotation
        cfg.update(workload="BASELINE.json configs[4]: 1000000 constant-product pools, 4096 tokens, Arbitrage(c=p), seed 3 "
                            "(the whole problem on the host cores at every N)", pools_total=M_POOLS, parallelism="host threads")
    return cfg


# --------------------------------------------------------------------------------------------------
def timed_steps(step, steps, warmup, barrier, clock_index, n_inst, preroll_ms=40.0):
    """W warm-up steps, then exactly `steps` steps replayed from CUDA graphs, CUDA-event timed, barrier + synchronize on
    both sides: a graph of CHUNK steps replayed steps // CHUNK times, then one graph of the steps % CHUNK left.  CHUNK is
    a multiple of 2 n_inst: every store is evaluated an even number of times per replay, so the ping-pong accumulator each
    call clears for the next one (PoolStore.evaluate) is the one the replayed graph starts from.  The clock sampler also
    covers a pre-roll of the CHUNK graph (the timed region itself is too short for NVML's sampling interval).
    Returns (ms_total, steps_timed, clocks, what the last timed step returned)."""
    import torch
    for i in range(max(warmup, 3)):
        step(i)
    barrier()
    CHUNK = max(1, 64 // (2 * n_inst)) * 2 * n_inst
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(min(n_inst, 64)):
            step(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(CHUNK):
            last = step(i)
    tail = None
    if steps % CHUNK:            # steps CHUNK * (steps // CHUNK) + i use instance i mod n_inst, as in the CHUNK graph
        tail = torch.cuda.CUDAGraph()
        with torch.cuda.graph(tail):
            for i in range(steps % CHUNK):
                last = step(i)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(clock_index) as clocks:
        barrier()
        # untimed pre-roll (clocks at their loaded value before the timed region).  A FIXED number of replays, the same on
        # every rank: the graphs contain the collective, so a time-based loop would let ranks replay different counts and
        # dead-lock in the all-reduce (it did, at N=4, this round).
        for _ in range(max(1, int(preroll_ms * 1e-3 / (12e-6 * CHUNK)))):
            graph.replay()
        torch.cuda.synchronize()
        barrier()
        torch.cuda.profiler.start()
        e0.record()
        for _ in range(steps // CHUNK):
            graph.replay()
        if tail is not None:
            tail.replay()
        e1.record()
        barrier()
        torch.cuda.profiler.stop()
    return e0.elapsed_time(e1), steps, clocks.summary(), last


def build_instances(I, cf, dev, rank, world, per, scaling, n_inst):
    """n_inst resident stores of `per` pools each + a price vector per store.  strong: store k is a 1/world slice of the
    1M-pool instance of seed 3 + 100 (k mod 8) -- this rank's own slice first, then the other slices, so that every rank
    holds n_inst different slabs; weak: `per` = 1M pools of this rank's own."""
    import torch
    f64 = dict(dtype=torch.float64, device=dev)
    stores, nus, hosts = [], [], {}
    for k in range(n_inst):
        base = k % 8
        if scaling == "weak":
            s = I.synth_const_product(per, N_TOKENS, seed=3 + 100 * base + 7919 * rank + 104729 * (k // 8))
        else:
            if base not in hosts:
                hosts[base] = I.synth_const_product(M_POOLS, N_TOKENS, seed=3 + 100 * base)
            s = hosts[base]
            sh = (rank + k // 8) % world
            sl = slice(sh * per, (sh + 1) * per)
            s = dict(s, idx=s["idx"][sl], reserves=s["reserves"][sl], gamma=s["gamma"][sl])
        hp = cf.HostPools.from_pairs(N_TOKENS, s["idx"], s["reserves"], s["gamma"])
        stores.append(cf.PoolStore(hp, device=dev, validate=False))
        nus.append(torch.as_tensor(s["prices"] * np.exp(0.01 * np.random.default_rng(k).standard_normal(N_TOKENS)), **f64))
    return stores, nus


def bench_configs(cf, I, dev):
    """BASELINE.json configs[0..3] through the public API on this GPU (time to a 1e-6 certificate, host buffers in),
    each beside the oracle on the host cores (bounded samples)."""
    import torch
    from oracle import cfmm_oracle as O
    out = []

    def gpu_solve(hp, util, **kw):
        best = None
        for _ in range(3):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            r = cf.solve_pools(hp, util, tol=1e-6, want_trades=False, device=dev, **kw)
            torch.cuda.synchronize(); w = time.perf_counter() - t0
            best = (w, r) if best is None or w < best[0] else best
        return best

    def entry(name, hp, util, o_util, full_oracle, **kw):
        w, r = gpu_solve(hp, util, **kw)
        e = {"config": name, "pools": int(hp.m), "n_tokens": int(hp.n_tokens), "time_to_1e-6_gap_ms": 1e3 * w,
             "solver_ms": 1e3 * r.wall_s, "status": r.status, "value_obj": r.value, "rel_gap": abs(r.gap),
             "primal_infeas": r.primal_infeas, "iters": r.iters, "evals": r.evals, "hvps": r.hvps,
             "value": hp.m * r.evals / w, "unit": UNIT}
        P = O.Pools(hp.n_tokens, hp.pool_ptr, hp.tok_idx, hp.reserves, hp.weights, hp.gamma, hp.kind)
        if full_oracle:
            t0 = time.perf_counter(); ro = O.solve(P, o_util, nu0=kw.get("nu0"), tol=1e-6); wo = time.perf_counter() - t0
            e["cpu_baseline"] = {"kind": "port", "cores": 1, "time_to_1e-6_gap_ms": 1e3 * wo, "value": hp.m * ro.evals / wo,
                                 "unit": UNIT, "sample": "oracle/cfmm_oracle.py::solve (numpy), whole solve",
                                 "value_obj": ro.value}
            e["obj_rel_diff_vs_oracle"] = abs(r.value - ro.value) / max(abs(ro.value), 1e-300)
        else:
            bk = O.Buckets(P); nu = np.asarray(kw.get("nu0") if kw.get("nu0") is not None else o_util.c, float)
            nu = np.where(nu > 0, nu, 1.0)
            O.evaluate(bk, nu)
            t0 = time.perf_counter(); k = 0
            while time.perf_counter() - t0 < 2.0:
                O.evaluate(bk, nu * (1 + 1e-3 * k)); k += 1
            wo = time.perf_counter() - t0
            e["cpu_baseline"] = {"kind": "port", "cores": 1, "value": hp.m * k / wo, "unit": UNIT,
                                 "sample": f"{k} oracle dual evaluations (numpy, oracle/cfmm_oracle.py::evaluate) in {wo:.1f}s"}
        out.append(e)

    d = I.arbitrage_instance()
    hp = cf.HostPools.from_lists(4, d["local_indices"], d["reserves"], d["fees"], d["kinds"], d["weights"])
    entry("configs[0] arbitrage.py as-is (5 pools, 4 tokens)", hp, cf.Arbitrage(d["market_value"]),
          O.Utility.arbitrage(d["market_value"]), True)
    s = I.synth_const_product(10_000, 256, seed=0)
    entry("configs[1] 10k constant-product pools, 256 tokens", cf.HostPools.from_pairs(256, s["idx"], s["reserves"], s["gamma"]),
          cf.Arbitrage(s["prices"]), O.Utility.arbitrage(s["prices"]), True)
    s = I.synth_mixed(100_000, 1000, seed=1)
    hp = cf.HostPools(1000, s["pool_ptr"], s["tok_idx"], s["reserves"], s["weights"], s["gamma"], s["kind"])
    entry("configs[2] 100k mixed pools (60% product, 30% weighted, 10% sum), 1k tokens", hp, cf.Arbitrage(s["prices"]),
          O.Utility.arbitrage(s["prices"]), False)
    s = I.synth_mixed(100_000, 1000, seed=2)
    hp = cf.HostPools(1000, s["pool_ptr"], s["tok_idx"], s["reserves"], s["weights"], s["gamma"], s["kind"])
    basket = I.synth_basket(1000, s["prices"], seed=2)
    entry("configs[3] liquidation.py objective (16-token basket -> token 0) over 100k mixed pools, 1k tokens", hp,
          cf.Liquidate(0, basket), O.Utility.liquidate(1000, 0, basket), False, nu0=s["prices"] / s["prices"][0])
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import cfmm_routing_code_b200 as cf
    from cfmm_routing_code_b200 import instances as I

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU leg")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    f64 = dict(dtype=torch.float64, device=dev)
    peer = world > 1 and args.collective == "peer"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(scaling):
        """the timed evaluation steps for one scaling mode: (ms_per_step, steps, clocks, eval-only ms_per_step, store, ...,
        the last timed step's [psi | arb] on the host)"""
        per = M_POOLS if scaling == "weak" else M_POOLS // world
        n_inst = n_instances(per)
        stores, nus = build_instances(I, cf, dev, rank, world, per, scaling, n_inst)
        use_peer = peer
        if use_peer:
            try:
                for st in stores:
                    st.enable_peer_allreduce()
            except Exception as e:                       # symmetric memory unavailable: NCCL does the all-reduce
                if rank == 0:
                    print(f"peer all-reduce unavailable ({type(e).__name__}: {e}); falling back to NCCL", file=sys.stderr)
                use_peer = False

        def step(i):
            acc = stores[i % n_inst].evaluate(nus[i % n_inst])      # peer mode: already all-reduced
            if world > 1 and not use_peer:
                dist.all_reduce(acc)
            return acc

        ms, steps, clocks, last = timed_steps(step, args.steps, args.warmup, barrier, local, n_inst)
        last = last.cpu().numpy()
        t = torch.tensor([ms], **f64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        eval_only = None
        if world > 1:            # the same steps without the collective: the all-reduce share of a step
            ms0, steps0, _, _ = timed_steps(lambda i: stores[i % n_inst].evaluate(nus[i % n_inst], reduce=False), args.steps,
                                            args.warmup, barrier, local, n_inst, preroll_ms=10.0)
            t0 = torch.tensor([ms0], **f64); dist.all_reduce(t0, op=dist.ReduceOp.MAX)
            eval_only = float(t0) / steps0
        return float(t) / steps, steps, clocks, eval_only, stores[0], per, n_inst, use_peer, last

    ms_per_step, steps, clocks, eval_only_ms, store0, per, n_inst, used_peer, last = measure(args.scaling)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "psi.npy"), np.asarray(last[:N_TOKENS], np.float64))
        np.save(os.path.join(args.dump_outputs, "arb.npy"), np.asarray(last[N_TOKENS:], np.float64))
    value = n_gpus * per / (ms_per_step * 1e-3)
    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_weak:
        torch.cuda.empty_cache()
        w_ms, w_steps, _, w_eval_only, _, w_per, w_inst, _, _ = measure("weak")
        weak = {"value": n_gpus * w_per / (w_ms * 1e-3), "unit": UNIT, "ms_per_step": w_ms, "pools_per_gpu": w_per,
                "pools_total": n_gpus * w_per, "eval_only_us": 1e3 * w_eval_only if w_eval_only else None,
                "allreduce_us": 1e3 * (w_ms - w_eval_only) if w_eval_only else None, "instances_per_gpu": w_inst}

    # ---- roofline of the dominant kernel: algorithmic bytes / avg launch duration
    alg_bytes = store0.algorithmic_bytes_per_eval()
    peak, peak_src = measured_peak()
    kernel_ms = eval_only_ms if eval_only_ms else ms_per_step
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tfile = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tfile) and per == M_POOLS:
        try:
            tj = json.load(open(tfile))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source", "profiles/traffic.json (ncu --set full capture of this kernel)")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": "k_blocked<eval> (csrc/cfmm_blocked.cu)",
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "note": "duration = timed region / steps (CUDA-graph replay of one kernel node per step" +
                        ("; the all-reduce share is excluded: eval-only replay of the same steps" if world > 1 else "") + ")"}

    # ---- e2e: the public API on HOST buffers: upload pools, solve to 1e-6, read psi/nu back
    e2e = None
    time_to_gap = None
    if not args.no_e2e:
        s = I.synth_const_product(M_POOLS, N_TOKENS, seed=3)
        hp = cf.HostPools.from_pairs(N_TOKENS, s["idx"], s["reserves"], s["gamma"]).pin_memory()
        util = cf.Arbitrage(s["prices"])
        cf.solve_pools(hp, util, tol=1e-6, want_trades=False, device=dev)      # warm-up (world > 1: creates the peer context once)
        runs = []
        for rep in range(E2E_REPS):
            barrier()
            t0 = time.perf_counter()
            r = cf.solve_pools(hp, util, tol=1e-6, want_trades=False, device=dev)      # world > 1: shards itself
            torch.cuda.synchronize()
            w = torch.tensor([time.perf_counter() - t0], **f64)
            if world > 1:
                dist.all_reduce(w, op=dist.ReduceOp.MAX)
            runs.append((float(w), r))
        runs.sort(key=lambda x: x[0])
        wall, r = runs[len(runs) // 2]                    # median of E2E_REPS (max over ranks each)
        h2d = (hp.reserves.nbytes + hp.tok_idx.nbytes + hp.gamma.nbytes) // max(world, 1) + 8 * 2 * N_TOKENS
        e2e = {"value": M_POOLS * r.evals / wall, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 16 * N_TOKENS + 64,
               "what": "cf.solve_pools(pinned host numpy pools, Arbitrage(p), tol=1e-6): upload (each rank its shard) + layout "
                       "build + native solve + psi/nu read-back; value = pools x dual evaluations / wall; median of %d" % E2E_REPS,
               "wall_s": wall, "wall_s_all": [x[0] for x in runs], "evals": r.evals, "hvps": r.hvps, "iters": r.iters,
               "status": r.status, "gap": r.gap, "primal_infeas": r.primal_infeas,
               "native_loop": r.info.history == []}
        time_to_gap = {"seconds_incl_upload": wall, "seconds_solver_only": r.wall_s, "rel_gap": abs(r.gap),
                       "primal_infeas": r.primal_infeas, "tol": 1e-6}

    cpu = None
    cfgs = None
    if rank == 0 and world == 1 and not args.no_cpu:
        data = _cfg5_host()
        v, k, dt, cores = cpu_eval_throughput(10.0, data)
        solve = cpu_full_solve(data)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "time_to_1e-6_gap_s": solve["wall_s"],
               "e2e_value": solve["value"],
               "sample": f"{k} oracle dual evaluations (C restatement, {cores} pthreads in a persistent pool, fp64) of the same "
                         f"1M-pool instance in {dt:.1f}s; time_to_1e-6_gap_s = oracle_solve_pairs (C Newton-PCG), best of 2"}
    if rank == 0 and world == 1 and not args.no_configs:
        cfgs = bench_configs(cf, I, dev)

    if rank == 0:
        cfgd = workload_config(n_gpus, args.scaling, n_inst)
        if world > 1:
            cfgd["collective_impl"] = ("cfmm_allreduce_ll: 16-byte {value, seq} pushes over NVLink peer memory, PDL-chained "
                                       "between the evaluation kernels" if used_peer else "NCCL all_reduce")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfgd, "roofline": roofline, "cpu_baseline": cpu,
            "e2e": e2e, "time_to_1e-6_gap": time_to_gap,
            "gpu_launches": steps * (2 if (world > 1 and used_peer) else 1), "clocks": clocks,
        }
        if world > 1:
            line["eval_only_us"] = 1e3 * eval_only_ms
            line["allreduce_us"] = 1e3 * (ms_per_step - eval_only_ms)
            line["weak"] = weak
        if cfgs is not None:
            line["configs"] = cfgs
        print(json.dumps(line), flush=True)
    if world > 1:
        sys.stdout.flush()
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)          # captured graphs + symmetric memory: skip the (hang-prone) communicator teardown


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 6400; --impl reference: 10)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 20; --impl reference: 1)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default, BASELINE configs[4]): 1M pools split over the GPUs; weak: 1M pools per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer solve leg (profiling runs)")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs[0..3] sub-lines")
    ap.add_argument("--no-weak", action="store_true", help="N>1: skip the secondary weak-scaled measurement")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="N>1: cfmm_allreduce_ll over NVLink peer memory (default) or NCCL all_reduce")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/psi.npy and DIR/arb.npy (float64)")
    args = ap.parse_args()
    reference = args.impl == "reference"
    if args.steps is None:                        # each reference step is seconds of CPU work
        args.steps = 10 if reference else 6400
    if args.warmup is None:
        args.warmup = 1 if reference else 20
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if reference and args.dump_outputs:
        ap.error("--dump-outputs writes the B200 path's outputs; it does not apply to --impl reference")
    # safety net: a wedged collective (a rank that died, a peer that never pushes) must end the run, not hold the box
    watchdog = threading.Timer(float(os.environ.get("CFMM_BENCH_WATCHDOG_S", "900")), lambda: os._exit(3))
    watchdog.daemon = True
    watchdog.start()
    if reference:
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
