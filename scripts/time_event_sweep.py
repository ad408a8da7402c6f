"""Wall clock of the event-based on-device closed loop (sweep.BatchedEventSweep): n = 5, N = 5, 4 event iterations, the
task-2 stop-and-go leader and time-headway policy (Sim_n_task_2), T = 50 timesteps, initial states from PlatoonEnv.reset
of seeds 0..S-1.

Arms, alternated within each batch size S = 10, 256, 4096: the fused glue kernel (groups launched in sequence, eager),
the torch glue (fused=False), the fused loop with the groups' eval and solve on forked streams, and the fused loop with
each iteration replayed as a CUDA graph.  Per arm one untimed full-size run, then the median of 3 timed runs.  At S = 10
also 10 serial fleet_event_based.simulate() calls, and pwa_friction (discrete gears) at n = 3, N = 3, S = 256, T = 10.
Each record gives the episode time, scenario-timesteps per second, and the fraction of scenario-iterations run after that
scenario stopped iterating (the reference's `break`): solve work that compacting active scenarios would save.  The
device name, power limit and max SM clock are read in the same run.
usage: python scripts/time_event_sweep.py OUT_DIR   (writes OUT_DIR/time_event_sweep.json)"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import hybrid_vehicle_platoon_b200 as hvp
from hybrid_vehicle_platoon_b200 import sweep as SW
from hybrid_vehicle_platoon_b200._sim import make_env_and_systems

ITERS = 4
ARMS = {"fused": dict(fused=True), "torch_glue": dict(fused=False), "fused_fork": dict(fused=True, fork=True),
        "fused_graph": dict(fused=True, graph=True)}
CASES = [("pwa_gear", 5, 5, 50, 10, list(ARMS)), ("pwa_gear", 5, 5, 50, 256, list(ARMS)),
         ("pwa_gear", 5, 5, 50, 4096, list(ARMS)), ("pwa_friction", 3, 3, 10, 256, ["fused"])]


def device_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def sim_for(model, n, N, T):
    sim = hvp.Sim_n_task_2(n, seed=0, N=N)
    sim.vehicle_model_type, sim.ep_len = model, T
    return sim


def initial_states(sim, S):
    env, _, _, _ = make_env_and_systems(sim, forward_real_ref=False)
    return np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                                dtype=np.float64).reshape(-1) for s in range(S)])


def timed(sim, ctx, x0, lx, T, arm):
    sw = SW.BatchedEventSweep(sim.n, sim.N, event_iters=ITERS, masses=sim.masses, spacing_policy=sim.spacing_policy,
                              model=sim.vehicle_model_type, ctx=ctx, **ARMS[arm])
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = sw.run(x0, lx, T)            # ends with a device synchronise and the read-back
        return time.perf_counter() - t0, r
    finally:
        sw.close()


def after_break(win):
    """Scenario-iterations run after the scenario's first iteration without a winner, over all scenario-iterations."""
    T, S, it = win.shape
    stop = np.where((win < 0).any(-1), (win < 0).argmax(-1), it - 1)
    return float((it - 1 - stop).sum() / (T * S * it))


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    out = sys.argv[1]
    os.makedirs(out, exist_ok=True)
    ctx = hvp.Context(0)
    res = dict(device=device_info(), workload=dict(iters=ITERS, leader="task-2 stop-and-go", policy="ConstantTimePolicy(10, 3)"),
               cases=[])
    print(res["device"], flush=True)
    for model, n, N, T, S, arms in CASES:
        sim = sim_for(model, n, N, T)
        lx = sim.leader_trajectory.get_leader_trajectory()
        x0 = initial_states(sim, S)
        for arm in arms:
            timed(sim, ctx, x0, lx, T, arm)      # full-size warm-up of every arm
        times = {a: [] for a in arms}
        outs = {}
        for _ in range(3):                        # the arms alternate
            for arm in arms:
                dt, r = timed(sim, ctx, x0, lx, T, arm)
                times[arm].append(dt)
                outs[arm] = r
        for arm in arms:
            med = float(np.median(times[arm]))
            r = outs[arm]
            row = dict(model=model, n=n, N=N, T=T, S=S, arm=arm, times_s=times[arm], median_s=med,
                       scenario_timesteps_per_s=S * T / med, after_break_fraction=after_break(r["winners"]),
                       mean_nodes=float(r["nodes"].mean()), infeasible=int((~r["feasible"]).sum()),
                       rollout_errors=int((r["errors"] != 0).sum()),
                       max_dX_vs_fused=float(np.nanmax(np.abs(r["X"] - outs[arms[0]]["X"]))),
                       winners_equal_fused=bool(np.array_equal(r["winners"], outs[arms[0]]["winners"])))
            res["cases"].append(row)
            print(json.dumps(row), flush=True)
        if S == 10:
            try:
                hvp.fleet_event_based.simulate(sim, event_iters=ITERS, seed=0, ep_len=T)    # warm-up of the host path
                t0 = time.perf_counter()
                for s in range(S):
                    hvp.fleet_event_based.simulate(sim, event_iters=ITERS, seed=s, ep_len=T)
                dt = time.perf_counter() - t0
                row = dict(model=model, n=n, N=N, T=T, S=S, arm="serial_simulate", calls=S, total_s=dt,
                           scenario_timesteps_per_s=S * T / dt)
            except (RuntimeError, RuntimeWarning) as e:    # simulate() raises where the sweep reports
                row = dict(model=model, n=n, N=N, T=T, S=S, arm="serial_simulate", error=repr(e))
            res["cases"].append(row)
            print(json.dumps(row), flush=True)
        with open(os.path.join(out, "time_event_sweep.json"), "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
