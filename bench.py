#!/usr/bin/env python
"""bench.py -- headline benchmark of the hybrid-MPC hot path (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--scenarios S] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): the per-vehicle local MIQPs of fleet_decent_mld.py /
fleet_seq_mld.py at n = 10 vehicles, horizon N = 6, pwa_gear model.  One STEP = one pass of the
hot path over one batch: S synthetic platoon scenarios x 10 vehicles = 10*S MIQPs, each solved to
proven optimality.  metric = hybrid-MPC solves/s (whole job, all GPUs).

    value : device-timed (CUDA events on the launching stream), inputs resident in HBM
    e2e   : same batch through the reference-facing C-ABI call with HOST (pinned) buffers,
            H2D + kernel + D2H inside the timed region
    roofline / fp64_pipe / rollout : how close the kernels run to the hardware
    cpu_baseline : the CPU oracle (exhaustive leaf enumeration, OpenMP) on a bounded sample

Under torchrun (N > 1) every rank runs the same per-GPU batch on its own seed (weak scaling, no
data-path collective: scenarios are independent); time = max over ranks.
"""
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

N_VEH, HORIZON = 10, 6
METRIC = "hybrid-MPC solves/sec at n=10,N=6 (per-vehicle local MIQPs, proven optimal)"


def make_batch(seed, scenarios):
    from hybrid_vehicle_platoon_b200.synth_local import platoon_local_problems
    rng = np.random.default_rng(seed)
    return platoon_local_problems(rng, scenarios, N_VEH, HORIZON)


def dump_outputs(out_dir, arrays, limit_bytes=64_000_000, seed=0):
    """Writes `arrays` (name -> CUDA tensor, first axis = problem) as <out_dir>/<name>.npy in float64, so that two builds
    can be compared output for output.  When they would exceed `limit_bytes` in all, every array keeps the same seeded
    sample of problems (in index order) and the sampled problem indices go to sample_index.npy."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    first = next(iter(arrays.values()))
    B = first.shape[0]
    row_bytes = 8 * sum(a[0].numel() for a in arrays.values())
    if B * row_bytes > limit_bytes:
        k = (limit_bytes - 4096) // (row_bytes + 8)          # 8 B per problem for the index; 4 KiB for the headers
        idx = np.sort(np.random.default_rng(seed).choice(B, k, replace=False))
        sel = torch.from_numpy(idx).to(first.device)
        arrays = {n: a.index_select(0, sel) for n, a in arrays.items()}
        np.save(os.path.join(out_dir, "sample_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.cpu().numpy().astype(np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(len(r) >= 6 and r[2 + k].startswith("Active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_reference_leg(scenarios_hint, budget_s=12.0, variants=True):
    """The CPU arm: the STRONGEST host implementation this repo has -- the product's own branch-and-bound compiled for
    the host (oracle/hvp_cpu_bnb.cpp, -O3 -march=native, built on this machine) under OpenMP over every core this
    process may use -- on a bounded sample of the bench workload.  `variants` adds the independent checker (exhaustive
    leaf enumeration, oracle/hvp_oracle.c) on a smaller sample, for scale.  Gurobi / dmpcpwa are not installable."""
    from oracle import oracle as O
    O.build()
    threads = O.use_all_cores()
    cal = make_batch(999, 64)
    args = lambda b: (HORIZON, b["flags"], b["mass"], b["x0"], b["xf"], b["xb"], b["xl"])
    O.local_miqp_bnb(*args(cal), native=True)                       # builds + warms
    t = time.perf_counter()
    O.local_miqp_bnb(*args(cal), native=True)
    per = (time.perf_counter() - t) / (64 * N_VEH)
    scen = int(max(64, min(scenarios_hint, budget_s / max(per, 1e-8) / N_VEH)))
    b = make_batch(1234 + 1, scen)
    t = time.perf_counter()
    r = O.local_miqp_bnb(*args(b), native=True)
    dt = time.perf_counter() - t
    assert (r["status"] == 2).all()
    out = {"value": scen * N_VEH / dt, "unit": "solves/s", "cores": int(r["threads"]), "kind": "port",
           "sample": f"{scen} scenarios x {N_VEH} vehicles (N={HORIZON}) of the bench distribution, {dt:.2f} s; "
                     f"port = the product's branch-and-bound (depth-first, dual-bound pruning, first dive; "
                     f"{float(r['nodes'].mean()):.1f} node QPs per solve) compiled for the host with -O3 -march=native, "
                     f"OpenMP over {int(r['threads'])} threads; the reference's solver (Gurobi behind dmpcpwa) is not "
                     f"installable here",
           "nodes_per_solve": float(r["nodes"].mean())}
    if variants:
        es = max(64, scen // 16)
        eb = make_batch(1234 + 1, es)
        t = time.perf_counter()
        ro = O.local_miqp(*args(eb))
        edt = time.perf_counter() - t
        out["variants"] = {"exhaustive_enumeration_checker": {
            "value": es * N_VEH / edt, "unit": "solves/s", "cores": threads, "leaves_per_solve": float(ro["leaves"].mean()),
            "what": "oracle/hvp_oracle.c: every reachable mode sequence x exact dual active-set QP (the independent "
                    "checker of the parity tests; -O2, OpenMP)"}}
    return out, dt, scen


def compiled_mpc_legs(hvp, torch, dev, stream, flush, steps=5, with_cpu=True):
    """BASELINE.json configs[0] and configs[2] on the compiled-MPC kernel (pm_kernel.cu): centralized
    MIQP n=3,N=5; naive-ADMM local MIQPs N=8; g-ADMM fixed-mode QPs N=8 -- device-timed, inputs in HBM."""
    from hybrid_vehicle_platoon_b200 import synth_mpc as G
    from oracle import oracle as O
    rng = np.random.default_rng(1234 + 2)
    legs = {}
    t = lambda a, dt=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to(dev).to(dt)

    def run(name, mpc, x0, params, fm=None, cpu=None):
        B, nl, N = x0.shape[0], mpc.n_local, mpc.N
        dx0, dm, dp = t(x0), t(np.full((B, nl), 800.0)), t(params)
        dfm = None if fm is None else t(fm, torch.int32)
        u = torch.empty(B, nl, N, dtype=torch.float64, device=dev)
        x = torch.empty(B, nl, 2, N + 1, dtype=torch.float64, device=dev)
        ex = torch.empty(B, max(mpc.n_extra, 1), dtype=torch.float64, device=dev)
        mo = torch.empty(B, nl, N, dtype=torch.int32, device=dev)
        ob = torch.empty(B, dtype=torch.float64, device=dev)
        st = torch.empty(B, dtype=torch.int32, device=dev)
        no = torch.empty(B, dtype=torch.int32, device=dev)
        it = torch.empty(B, dtype=torch.int32, device=dev)
        ms = []
        for i in range(2 + steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            mpc.solve_device(B, dx0, dm, dp, dfm, u, x, ex, mo, ob, st, no, it, stream=stream)
            b.record()
            flush.fill_(1)
            torch.cuda.synchronize()
            if i >= 2:
                ms.append(a.elapsed_time(b))
        leg = {"value": B / (np.mean(ms) * 1e-3), "unit": "solves/s", "batch": B, "ms_per_launch": float(np.mean(ms)),
               "variables": mpc.n_var, "nodes_per_solve": float(no.double().mean()),
               "qp_iters_per_solve": float(it.double().mean()), "optimal_frac": float((st == 2).double().mean())}
        if cpu is not None and with_cpu:
            t0 = time.perf_counter()
            cpu()
            leg["cpu_port_solves_per_s"] = cpu.count / (time.perf_counter() - t0)
            leg["cpu_port"] = f"oracle branch-and-bound + exact QP, OpenMP over {O.max_threads()} threads, {cpu.count} problems"
        legs[name] = leg

    class _Cpu:
        def __init__(self, count, fn):
            self.count, self.fn = count, fn

        def __call__(self):
            self.fn(self.count)

    B = 16384
    x0, params = G.cent_cases(rng, B, 3, 5)
    run("cent_n3_N5 (configs[0]: MpcMldCent MIQP)", hvp.api.CompiledMpc(G.CENT, 5, n_local=3), x0, params,
        cpu=_Cpu(512, lambda c: O.mpc_solve(O.CENT, 3, 5, x0[:c], 800.0, params[:c], method=1)))
    x0, params = G.admm_cases(rng, B, 8)
    run("naive_admm_local_N8 (configs[2]: LocalMpcADMM MIQP, interior vehicle)", hvp.api.CompiledMpc(G.ADMM, 8, rho=0.5),
        x0, params, cpu=_Cpu(512, lambda c: O.mpc_solve(O.ADMM, 1, 8, x0[:c], 800.0, params[:c], rho=0.5, method=1)))
    x0, params, fm = G.gadmm_cases(rng, 4 * B, 1, 1, 8)
    run("g_admm_fixed_mode_qp_N8 (configs[2]: local fixed-mode QPs per ADMM round)",
        hvp.api.CompiledMpc(G.GADMM, 8, n_front=1, n_behind=1, rho=0.5), x0, params, fm=fm,
        cpu=_Cpu(4096, lambda c: O.mpc_solve(O.GADMM, 1, 8, x0[:c], 800.0, params[:c], n_front=1, n_behind=1, rho=0.5,
                                             fixed_modes=fm[:c])))
    # 1-norm (MILP) variant, quadratic_cost=False (SURVEY.md 8f rank 3): LP node problems by proximal-point rounds
    x0, params = G.cent_cases(rng, 512, 3, 5)
    run("cent_n3_N5_one_norm (configs[0] shape, MILP: quadratic_cost=False)",
        hvp.api.CompiledMpc(G.CENT, 5, n_local=3, one_norm=True), x0, params)
    from hybrid_vehicle_platoon_b200.synth_local import platoon_local_problems
    c = platoon_local_problems(rng, 2048, N_VEH, HORIZON)
    sel = np.nonzero(c["flags"] == 0)[0]
    pl = np.concatenate([c[k][sel].reshape(len(sel), -1) for k in ("xf", "xb", "xl")], axis=1)
    run("local_n10_N6_one_norm (configs[1] shape, interior vehicles, MILP: quadratic_cost=False)",
        hvp.api.CompiledMpc(G.LOCAL, HORIZON, flags=0, one_norm=True), c["x0"][sel].reshape(-1, 1, 2), pl)
    return legs


def _episodes(run, reps=3, sync=None, reduce=None):
    """Wall-clock time of a whole-episode leg: one untimed run at FULL size first (the CPU-side work of the previous leg
    leaves the GPU at idle clocks and the caching allocator without blocks of this size: measured 55 ms for the first
    runs of the decentralized loop against 40-43 ms from the third on, scripts/diag_decent_loop.py), then the MEDIAN of
    `reps` timed runs; every run includes the upload of the initial states and the read-back of all result arrays."""
    run()
    times, out = [], None
    for _ in range(reps):
        if sync:
            sync()
        t0 = time.perf_counter()
        out = run()
        dt = time.perf_counter() - t0
        times.append(reduce(dt) if reduce else dt)
    return out, sorted(times)[len(times) // 2], times


def closed_loop_leg(ctx, S=4096, T=20):
    """Whole closed-loop episodes of the decentralized controller for S scenarios, state resident on the device
    (sweep.BatchedDecentSweep): observe -> S*n MIQPs -> rollout per timestep, wall-clock incl. result read-back."""
    from hybrid_vehicle_platoon_b200.sweep import BatchedDecentSweep
    from hybrid_vehicle_platoon_b200.misc import StopAndGoLeaderTrajectory
    rng = np.random.default_rng(1234 + 3)
    v = np.floor(rng.uniform(5, 35, (S, N_VEH))); gaps = rng.uniform(60, 160, (S, N_VEH))
    p = np.floor(3000.0 - np.cumsum(gaps, 1) + gaps[:, :1])
    x0 = np.empty((S, 2 * N_VEH)); x0[:, 0::2] = p; x0[:, 1::2] = v
    lx = StopAndGoLeaderTrajectory(p=3000, vh=20, vl=10, vf=30, v_change_steps=[5, 12], trajectory_len=T + HORIZON + 10,
                                   ts=1).get_leader_trajectory()
    sw = BatchedDecentSweep(N_VEH, HORIZON, ctx=ctx)
    out, dt, runs = _episodes(lambda: sw.run(x0, lx, T))
    return {"value": S * T / dt, "unit": "scenario-timesteps/s", "solves_per_s": S * T * N_VEH / dt, "scenarios": S,
            "timesteps": T, "seconds": dt, "seconds_runs": runs, "optimal_frac": float((out["status"] == 2).mean()),
            "rollout_exceptions": int((out["errors"] != 0).any(0).sum()),
            "mean_nodes": float(out["nodes"].mean())}


def admm_loop_leg(ctx, S=1024, T=2, n=15, N=8, iters=20):
    """BASELINE.json configs[2]: naive-ADMM consensus rounds at n = 15, N = 8 for S scenarios on the device
    (sweep.BatchedAdmmSweep): per round the S*n local MIQPs are three launches (front / interior / trailer)."""
    from hybrid_vehicle_platoon_b200.sweep import BatchedAdmmSweep
    from hybrid_vehicle_platoon_b200.misc import ConstantVelocityLeaderTrajectory
    rng = np.random.default_rng(1234 + 2)
    v = np.floor(rng.uniform(10, 30, (S, n))); gaps = rng.uniform(60, 140, (S, n))
    p = np.floor(3000.0 - np.cumsum(gaps, 1) + gaps[:, :1])
    x0 = np.empty((S, 2 * n)); x0[:, 0::2] = p; x0[:, 1::2] = v
    lx = ConstantVelocityLeaderTrajectory(p=3000, v=20, trajectory_len=T + N + 10, ts=1).get_leader_trajectory()
    sw = BatchedAdmmSweep(n, N, admm_iters=iters, rho=0.5, ctx=ctx)
    out, dt, runs = _episodes(lambda: sw.run(x0, lx, T))
    return {"value": S * T * iters / dt, "unit": "scenario-ADMM-rounds/s", "solves_per_s": S * T * iters * n / dt,
            "scenarios": S, "timesteps": T, "admm_iters": iters, "seconds": dt, "seconds_runs": runs,
            "optimal_frac": float((out["status"] == 2).mean()), "rollout_exceptions": int((out["errors"] != 0).any(0).sum())}


def gadmm_loop_leg(ctx, S=1024, T=2, n=15, N=8, iters=100):
    """BASELINE.json configs[2], the convex half: switching ("g") ADMM at n = 15, N = 8 for S scenarios on the device
    (sweep.BatchedGAdmmSweep): per round the S*n fixed-mode QPs are one launch per role through the FP64 tensor-core
    precompute, z / y updates and the re-identification of the mode sequences are torch ops; up to two warm starts per
    timestep, 100 rounds each (fleet_g_admm.py:255-301, :405)."""
    from hybrid_vehicle_platoon_b200.sweep import BatchedGAdmmSweep
    from hybrid_vehicle_platoon_b200.misc import ConstantVelocityLeaderTrajectory
    rng = np.random.default_rng(1234 + 2)
    v = np.floor(rng.uniform(12, 28, (S, n))); gaps = rng.uniform(60, 120, (S, n))
    p = np.floor(3000.0 - np.cumsum(gaps, 1) + gaps[:, :1])
    x0 = np.empty((S, 2 * n)); x0[:, 0::2] = p; x0[:, 1::2] = v
    lx = ConstantVelocityLeaderTrajectory(p=3000, v=20, trajectory_len=T + N + 10, ts=1).get_leader_trajectory()
    sw = BatchedGAdmmSweep(n, N, admm_iters=iters, rho=0.5, ctx=ctx)
    sw.run(x0[:16], lx, 1)
    out, dt, runs = _episodes(lambda: sw.run(x0, lx, T))
    rounds = S * iters * (1 + 2 * (T - 1))            # one warm start at t = 0, two afterwards
    return {"value": rounds / dt, "unit": "scenario-ADMM-rounds/s", "qp_solves_per_s": rounds * n / dt, "scenarios": S,
            "timesteps": T, "admm_iters": iters, "seconds": dt, "seconds_runs": runs, "solved_frac": float(out["solved"].mean()),
            "rollout_exceptions": int((out["errors"] != 0).any(0).sum())}


def mixed_sweep_leg(ctx, rank, world, dev, S=4096, T=10):
    """BASELINE.json configs[3]: Monte-Carlo sweep of S synthetic platoon scenarios with n ~ U{5..15}, N ~ U{4..10},
    stop-and-go leader with random change steps / speeds, 50/50 constant spacing vs time headway (SURVEY 8d), whole
    closed loops of the decentralized controller on the device.  EVERY rank calls this: the scenarios are dealt to the
    ranks by the 7 n N cost proxy (dist.balanced_shards), no collective on the data path; time = max over ranks."""
    import torch
    from hybrid_vehicle_platoon_b200.dist import max_over_ranks, sum_over_ranks
    from hybrid_vehicle_platoon_b200.misc import ConstantSpacingPolicy, ConstantTimePolicy, StopAndGoLeaderTrajectory
    from hybrid_vehicle_platoon_b200.sweep import run_mixed_sweep
    rng = np.random.default_rng(1234 + 3)            # the same scenario list on every rank
    scen = []
    for _ in range(S):
        n, N = int(rng.integers(5, 16)), int(rng.integers(4, 11))
        v = np.floor(rng.uniform(8, 30, n)); gaps = rng.uniform(60, 160, n)
        p = np.floor(3000.0 - np.cumsum(gaps) + gaps[0])
        x0 = np.empty(2 * n); x0[0::2] = p; x0[1::2] = v
        lx = StopAndGoLeaderTrajectory(p=3000, vh=20, vl=float(rng.uniform(8, 14)), vf=float(rng.uniform(22, 32)),
                                       v_change_steps=[int(rng.integers(2, 5)), int(rng.integers(5, 9))],
                                       trajectory_len=T + 10 + 12, ts=1).get_leader_trajectory()
        pol = ConstantSpacingPolicy(50) if rng.random() < 0.5 else ConstantTimePolicy(10, 3)
        scen.append(dict(n=n, N=N, x0=x0, leader_x=lx, masses=None, spacing_policy=pol))
    def sync():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def run():
        r = run_mixed_sweep(scen, T, rank=rank, world=world, device=dev.index, ctx=ctx)
        torch.cuda.synchronize()
        return r

    out, dt, runs = _episodes(run, sync=sync, reduce=lambda d: max_over_ranks([d], device=dev)[0])
    solves = sum(scen[i]["n"] for i in out) * T
    opt = sum(int((r["status"] == 2).sum()) for r in out.values())
    tot_s, tot_o, tot_n = sum_over_ranks([solves, opt, len(out)], device=dev)
    return {"value": S * T / dt, "unit": "scenario-timesteps/s", "solves_per_s": tot_s / dt, "scenarios": int(tot_n),
            "timesteps": T, "seconds": dt, "seconds_runs": runs, "optimal_frac": tot_o / max(tot_s, 1), "n_range": [5, 15], "N_range": [4, 10],
            "sharding": "dist.balanced_shards by 7 n N, no data-path collective", "n_gpus": world}


def tree_split_leg(ctx, dev, n=8, N=6, problems=4, depth=0, groups=256, stress=False, seed=5):
    """ONE large centralized MIQP tree (n = 8, N = 6: 48 variables) searched by all ranks together: every rank takes
    the sub-trees whose mode-prefix ordinal is congruent to its rank, the incumbent bound is exchanged with an NCCL
    allreduce(min) (dist.solve_tree_split).  EVERY rank calls this; time = CUDA events, max over ranks."""
    import torch
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import dist as D
    from hybrid_vehicle_platoon_b200 import synth_mpc as G
    rng = np.random.default_rng(seed)
    x0, params = G.cent_cases(rng, problems, n, N, stress=stress)
    mpc = hvp.api.CompiledMpc(G.CENT, N, n_local=n, ctx=ctx)
    tx0 = torch.as_tensor(x0, device=dev); tp = torch.as_tensor(params, device=dev)
    tm = torch.full((problems, n), 800.0, dtype=torch.float64, device=dev)
    ms, out = [], None
    for rep in range(3):
        D.dist_allreduce(torch.zeros(1, device=dev), "sum")           # line the ranks up
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = D.solve_tree_split(mpc, tx0, tm, tp, groups=groups, prefix_depth=depth)
        b.record()
        torch.cuda.synchronize()
        if rep > 0:
            ms.append(D.max_over_ranks([a.elapsed_time(b)], device=dev)[0])
    return {"value": problems / (float(np.mean(ms)) * 1e-3), "unit": "solves/s", "ms": float(np.mean(ms)), "problems": problems,
            "variables": n * N, "prefix_depth": depth if depth else "library default (n + 2 on one device, two more levels per doubling of the world)", "warps_per_problem_per_gpu": groups,
            "optimal_frac": float((out["status"] == 2).double().mean()), "nodes_per_solve": float(out["nodes"].double().mean()),
            "collective": "allreduce(min) of the incumbent objective, 8 B per problem, twice per solve (one device: none)"}


def workload_config(S):
    """`config` of the headline workload -- identical in both arms (the reference arm times bounded samples of it)."""
    return {"workload": f"fleet_decent_mld.py per-vehicle local MIQPs (LocalMpcMld, pwa_gear), n={N_VEH}, N={HORIZON}; "
                        f"{S} scenarios x {N_VEH} vehicles = {S * N_VEH} MIQPs per GPU per step, reference reset "
                        f"distribution, constant-velocity neighbour predictions, gap 0 (proven optimal)",
            "scenarios_per_gpu": S, "n": N_VEH, "N": HORIZON}


def full_config(S):
    """Byte-identical in both arms; what differs per arm (the GPU arm's L2 flush, the CPU arm's bounded sample) is
    described in the same words on both sides."""
    return dict(workload_config(S),
                timing="b200 arm: L2 flushed (256 MiB write) between timed steps, steps timed individually with CUDA "
                       "events; reference arm: each step is a bounded sample of the same workload on the host cores "
                       "(see cpu_baseline.sample)")


def run_reference(args, rank, world):
    if rank != 0:
        return
    times, solves = [], 0
    base = first = None
    for i in range(args.warmup + args.steps):
        base, dt, scen = cpu_reference_leg(args.scenarios, budget_s=3.0, variants=(i == 0))
        first = first or base
        if i >= args.warmup:
            times.append(dt)
            solves += scen * N_VEH
    val = solves / sum(times)
    base["value"] = val
    if first and "variants" in first:
        base["variants"] = first["variants"]
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "solves/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": full_config(args.scenarios),
            "cpu_baseline": base,
            "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_JSON_FD = None


def emit(obj):
    """The ONE JSON line of the contract, written to the process's ORIGINAL stdout."""
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    # stdout must carry exactly one JSON line, but native libraries print there too (NCCL writes its version banner
    # to fd 1 from C, whatever NCCL_DEBUG says): keep a private copy of the original stdout for the JSON line and
    # point fd 1 at stderr for everything else.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scenarios", type=int, default=65536, help="platoon scenarios per GPU per step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--profile", action="store_true",
                    help="short run for ncu: device-timed MIQP steps + rollout launches only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the solutions of the last timed step (u, x, modes, obj, status; rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the ONE JSON line: NCCL prints its version banner to stdout at NCCL_DEBUG=VERSION
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    ctx = hvp.Context(local_rank)
    S, B = args.scenarios, args.scenarios * N_VEH
    batch = make_batch(1234 + 1 + 7919 * rank, S)

    # ---- device-resident inputs / outputs ----
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_flags, d_mass, d_x0 = t(batch["flags"]), t(batch["mass"]), t(batch["x0"])
    d_xf, d_xb, d_xl = t(batch["xf"]), t(batch["xb"]), t(batch["xl"])
    d_u = torch.empty((B, HORIZON), dtype=torch.float64, device=dev)
    d_x = torch.empty((B, 2, HORIZON + 1), dtype=torch.float64, device=dev)
    d_modes = torch.empty((B, HORIZON), dtype=torch.int32, device=dev)
    d_obj = torch.empty(B, dtype=torch.float64, device=dev)
    d_status = torch.empty(B, dtype=torch.int32, device=dev)
    d_nodes = torch.empty(B, dtype=torch.int32, device=dev)
    d_iters = torch.empty(B, dtype=torch.int32, device=dev)
    desc = api.local_desc(HORIZON)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def step_dev():
        api.local_miqp_device(desc, B, d_flags, d_mass, d_x0, d_xf, d_xb, d_xl, d_u, d_x, d_modes, d_obj,
                              d_status, d_nodes, d_iters, ctx=ctx, stream=stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = ctx.launch_count
    for _ in range(args.warmup):
        step_dev()
        flush.fill_(1)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches_t0 = ctx.launch_count
    for a, b_ in ev:
        a.record()
        step_dev()
        b_.record()
        flush.fill_(1)          # L2 flush between timed steps (outside the event pairs)
    barrier()
    launches_timed = ctx.launch_count - launches_t0
    ms = np.array([a.elapsed_time(b_) for a, b_ in ev])
    total_ms = float(ms.sum())
    assert bool((d_status == 2).all()), "a bench problem was not solved to optimality"
    if args.dump_outputs and rank == 0:
        # node and QP-iteration counts are left out: which worker adopts which sub-tree depends on scheduling
        dump_outputs(args.dump_outputs, {"u": d_u, "x": d_x, "modes": d_modes, "obj": d_obj, "status": d_status})
    nodes_mean = float(d_nodes.double().mean())
    iters_mean = float(d_iters.double().mean())

    if args.profile:
        rb = 1 << 20
        rng = np.random.default_rng(4321)
        v = rng.uniform(6, 33, (rb, N_VEH)); gaps = rng.uniform(30, 150, (rb, N_VEH))
        p = 3000.0 - np.cumsum(gaps, 1)
        xs = np.empty((rb, 2 * N_VEH)); xs[:, 0::2] = p; xs[:, 1::2] = v
        rx = t(xs); ru = t(rng.uniform(-1, 1, (rb, N_VEH)))
        rg = t(np.clip(np.digitize(v, [9.235, 12.855, 16.93, 23.315, 32.47]) + 1, 1, 6).astype(np.int32))
        rm = t(rng.uniform(700, 1000, (rb, N_VEH)))
        rl = t(np.stack([p[:, 0] + 5, np.full(rb, 20.0)], 1))
        rxo = torch.empty_like(rx); rc = torch.empty(rb, dtype=torch.float64, device=dev)
        rv = torch.empty(rb, dtype=torch.uint8, device=dev); re_ = torch.empty(rb, dtype=torch.int32, device=dev)
        rdesc = api.env_desc(N_VEH, mass_per_scenario=True)
        for i in range(args.steps):
            api.rollout_step_device(rdesc, rb, rx, ru, rg, rm, rl, rxo, rc, rv, re_, ctx=ctx, stream=stream)
            flush.fill_(1)
        torch.cuda.synchronize()
        emit({"profile_run": True, "ms_per_step": float(ms.mean()), "solves_per_s": B / (ms.mean() * 1e-3),
              "nodes_per_solve": nodes_mean, "qp_iters_per_solve": iters_mean})
        return

    # ---- e2e: reference-facing host call with pinned host buffers ----
    def pinned(a):
        tt = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return tt, tt.numpy()
    keep = []
    h = {}
    for k in ("flags", "mass", "x0", "xf", "xb", "xl"):
        tt, h[k] = pinned(batch[k]); keep.append(tt)
    ho = {}
    for k, shape, dt in (("u", (B, HORIZON), np.float64), ("x", (B, 2, HORIZON + 1), np.float64),
                         ("modes", (B, HORIZON), np.int32), ("obj", (B,), np.float64),
                         ("status", (B,), np.int32), ("nodes", (B,), np.int32)):
        tt, ho[k] = pinned(np.empty(shape, dt)); keep.append(tt)
    import ctypes as C
    hp = lambda a: a.ctypes.data_as(C.c_void_p)
    L = hvp._lib.lib()

    def step_host():
        hvp._lib.check(L.hvp_local_miqp_host(ctx.handle, C.byref(desc), B, hp(h["flags"]), hp(h["mass"]),
                                             hp(h["x0"]), hp(h["xf"]), hp(h["xb"]), hp(h["xl"]), hp(ho["u"]),
                                             hp(ho["x"]), hp(ho["modes"]), hp(ho["obj"]), hp(ho["status"]),
                                             hp(ho["nodes"]), None))
    h2d = sum(h[k].nbytes for k in h)
    d2h = sum(ho[k].nbytes for k in ho)
    for _ in range(3):
        step_host()
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert np.array_equal(ho["status"], d_status.cpu().numpy())
    # the same call on PAGEABLE numpy arrays (what a maintainer's script holds): the copies are staged by the driver
    hpg = {k: np.array(batch[k], copy=True) for k in ("flags", "mass", "x0", "xf", "xb", "xl")}
    hog = {k: np.empty_like(v) for k, v in ho.items()}

    def step_host_pageable():
        hvp._lib.check(L.hvp_local_miqp_host(ctx.handle, C.byref(desc), B, hp(hpg["flags"]), hp(hpg["mass"]),
                                             hp(hpg["x0"]), hp(hpg["xf"]), hp(hpg["xb"]), hp(hpg["xl"]), hp(hog["u"]),
                                             hp(hog["x"]), hp(hog["modes"]), hp(hog["obj"]), hp(hog["status"]),
                                             hp(hog["nodes"]), None))
    step_host_pageable()
    pg_steps = 3
    t0 = time.perf_counter()
    for _ in range(pg_steps):
        step_host_pageable()
    torch.cuda.synchronize()
    pg_s = time.perf_counter() - t0
    assert np.array_equal(hog["status"], ho["status"])
    # the host path (chunks) and the device path (one launch) agree to round-off: which lane solves a leaf in the tail
    # of a launch depends on the launch shape (sub-tree adoption, DESIGN 2.2)
    assert np.allclose(ho["obj"], d_obj.cpu().numpy(), rtol=1e-9, atol=0)
    clocks = sampler.stop()

    # ---- max over ranks ----
    from hybrid_vehicle_platoon_b200.dist import max_over_ranks
    total_ms, e2e_s, pg_s = max_over_ranks([total_ms, e2e_s, pg_s], device=dev)
    value = world * B * args.steps / (total_ms * 1e-3)
    e2e_value = world * B * e2e_steps / e2e_s
    e2e_pageable = world * B * pg_steps / pg_s

    # ---- legs that every rank takes part in ----
    shared_legs = {}
    if not args.profile:
        shared_legs["mixed_sweep_n5-15_N4-10 (configs[3]: 4096 scenarios sharded over the GPUs, on-device closed loops)"] = \
            mixed_sweep_leg(ctx, rank, world, dev)
        shared_legs["tree_split_cent_n8_N6 (one large MIQP tree searched by all GPUs, allreduce-min of the incumbent)"] = \
            tree_split_leg(ctx, dev)
        shared_legs["tree_split_cent_n10_N6 (the centralized size BASELINE.json's metric names: 60 variables)"] = \
            tree_split_leg(ctx, dev, n=10, N=6)

    out = None
    if rank == 0:
        hbm_peak, peak_src = peaks()
        bytes_per_solve = 4 + 8 + 16 + 3 * 16 * (HORIZON + 1) + 8 * HORIZON + 16 * (HORIZON + 1) + 4 * HORIZON + 8 + 4 + 4 + 4
        kern_ms = total_ms / args.steps
        achieved = B * bytes_per_solve / (kern_ms * 1e-3) / 1e9
        # FP64 work model (DESIGN.md): flops per node (build + factor + objective) and per active-set iteration
        n = HORIZON
        f_node = 2 * n * n + n ** 3 / 3 + 2 * n ** 3 + 2 * n * n + 4 * n * n
        f_iter = 14 * n + 2 * n * n + 2 * n * n + n ** 3 / 3 + 2 * n * n + 2 * n * n + 2 * n * n
        flops_per_solve = nodes_mean * f_node + iters_mean * f_iter
        peak_clk0 = ClockSampler(local_rank)
        peak_clk0.start()
        fp64_peak = hvp.microbench_fp64(20000, ctx=ctx)
        fp64_ach = B * flops_per_solve / (kern_ms * 1e-3) / 1e12

        # ---- rollout kernel (c): HBM-bound, 1M scenario-steps ----
        rb = 1 << 20
        rng = np.random.default_rng(4321)
        v = rng.uniform(6, 33, (rb, N_VEH)); gaps = rng.uniform(30, 150, (rb, N_VEH))
        p = 3000.0 - np.cumsum(gaps, 1)
        xs = np.empty((rb, 2 * N_VEH)); xs[:, 0::2] = p; xs[:, 1::2] = v
        rx = t(xs); ru = t(rng.uniform(-1, 1, (rb, N_VEH)))
        rg = t(np.clip(np.digitize(v, [9.235, 12.855, 16.93, 23.315, 32.47]) + 1, 1, 6).astype(np.int32))
        rm = t(rng.uniform(700, 1000, (rb, N_VEH)))
        rl = t(np.stack([p[:, 0] + 5, np.full(rb, 20.0)], 1))
        rxo = torch.empty_like(rx); rc = torch.empty(rb, dtype=torch.float64, device=dev)
        rv = torch.empty(rb, dtype=torch.uint8, device=dev); re_ = torch.empty(rb, dtype=torch.int32, device=dev)
        rdesc = api.env_desc(N_VEH, mass_per_scenario=True)
        rms = []
        for i in range(args.warmup + args.steps):
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            api.rollout_step_device(rdesc, rb, rx, ru, rg, rm, rl, rxo, rc, rv, re_, ctx=ctx, stream=stream)
            b_.record()
            flush.fill_(1)
            torch.cuda.synchronize()
            if i >= args.warmup:
                rms.append(a.elapsed_time(b_))
        r_ms = float(np.mean(rms))
        r_bytes = 52 * N_VEH + 29
        r_ach = rb * r_bytes / (r_ms * 1e-3) / 1e9
        rollout = {"metric": "rollout scenario-steps/s (n=10, given gears, per-scenario masses)",
                   "value": rb / (r_ms * 1e-3), "unit": "scenario-steps/s", "ms_per_launch": r_ms,
                   "batch": rb, "errors": int((re_ != 0).sum()),
                   "roofline": {"bound": "hbm", "achieved": r_ach, "peak": hbm_peak, "unit": "GB/s",
                                "frac": r_ach / hbm_peak,
                                # dram__bytes_read.sum + dram__bytes_write.sum of this launch shape, ncu --set full
                                # (profiles/r01g_rollout_ncu_raw.csv; the kernel has not changed since)
                                "traffic": 552.4e6 if rb == (1 << 20) else None, "traffic_unit": "bytes per launch (ncu)",
                                "algorithmic_bytes_per_scenario_step": r_bytes, "peak_source": peak_src}}

        # ---- p99 per-timestep latency: one scenario (10 MIQPs) through the host call ----
        # (SURVEY 8d: >= 10^4 timesteps; every call is a DIFFERENT scenario of the bench distribution)
        pool = make_batch(77, 512)
        sl = lambda a, j: a[j * N_VEH:(j + 1) * N_VEH]
        lat = []
        for i in range(10200):
            j = i % 512
            t0 = time.perf_counter()
            hvp.local_miqp(HORIZON, sl(pool["flags"], j), sl(pool["mass"], j), sl(pool["x0"], j), sl(pool["xf"], j),
                           sl(pool["xb"], j), sl(pool["xl"], j), ctx=ctx)
            lat.append(time.perf_counter() - t0)
        lat = np.array(lat[200:]) * 1e3
        smem_peak = hvp.api.microbench_smem(20000, ctx)
        for _ in range(20):                  # long enough for the clock sampler to see the microbenchmarks under load
            hvp.microbench_fp64(20000, ctx=ctx)
            hvp.api.microbench_smem(20000, ctx)
        peak_clocks = peak_clk0.stop()

        cpu = None
        if not args.no_cpu:
            cpu, _, _ = cpu_reference_leg(S, budget_s=12.0)
        other = compiled_mpc_legs(hvp, torch, dev, stream, flush, with_cpu=not args.no_cpu)
        other.update(shared_legs)
        other["closed_loop_decent_n10_N6 (configs[3] shape: 4096 scenarios, on-device episode)"] = closed_loop_leg(ctx)
        other["closed_loop_naive_admm_n15_N8 (configs[2]: 1024 scenarios x 20 ADMM rounds per timestep)"] = admm_loop_leg(ctx)
        other["closed_loop_g_admm_n15_N8 (configs[2]: 1024 scenarios x 100 ADMM rounds x <= 2 warm starts per timestep)"] = gadmm_loop_leg(ctx)

        out = {
            "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": full_config(S),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "call": "hvp_local_miqp_host (pinned numpy in, numpy out)",
                    "pageable_value": e2e_pageable,
                    "pageable_note": "same call on ordinary (pageable) numpy arrays, 3 steps",
                    # the other half of BASELINE.json's metric: one scenario-timestep (10 MIQPs) through the same host call
                    "latency_p50_ms": float(np.percentile(lat, 50)), "latency_p99_ms": float(np.percentile(lat, 99))},
            "gpu_launches": int(launches_timed),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch of 655 360 solves, ncu --set full
                         # (profiles/r01o_flat_ncu_raw.csv): 517 B per solve against 568 algorithmic
                         "traffic": 338.67e6 * (B / 655360.0), "traffic_unit": "bytes per launch (ncu, scaled by the batch)",
                         "algorithmic_bytes_per_solve": bytes_per_solve, "peak_source": peak_src,
                         "kernel": "flat_miqp_kernel<6>",
                         "note": "on-chip FP64 branch-and-bound: HBM traffic is parameters in + solution "
                                 "out only, so the HBM fraction is small by construction; see fp64_pipe"},
            "fp64_pipe": {"achieved_tflops": fp64_ach, "peak_tflops": fp64_peak, "frac": fp64_ach / fp64_peak,
                          "peak_source": "hvp_microbench_fp64 (measured DFMA issue peak)", "peak_clocks": peak_clocks,
                          "flops_per_solve_model": flops_per_solve, "nodes_per_solve": nodes_mean,
                          "qp_iters_per_solve": iters_mean},
            "latency": {"what": "one scenario-timestep = 10 local MIQPs through hvp_local_miqp_host (host buffers in, "
                                "controls out), a different scenario per call; 8 workers per tree (coop_split_kernel)",
                        "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)),
                        "max_ms": float(lat.max()), "samples": int(lat.size),
                        "full_batch": {"what": f"{S} scenario-timesteps per launch (device-timed steps above)",
                                       "p50_ms": float(np.percentile(ms, 50)), "max_ms": float(np.max(ms)),
                                       "samples": int(ms.size)}},
            "smem": {"peak_gbs": smem_peak, "peak_source": "hvp_microbench_smem (measured LDS.128 read bandwidth, whole device)",
                     "peak_clocks": peak_clocks,
                     "note": "achieved shared-memory traffic of the QP kernels is read from ncu "
                             "(l1tex__data_pipe_lsu_wavefronts_mem_shared, profiles/README.md)"},
            "rollout": rollout,
            "other_configs": other,
            "cpu_baseline": cpu,
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        emit(out)


if __name__ == "__main__":
    main()
