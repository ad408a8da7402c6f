"""Wall clock of the centralized on-device closed loop (sweep.BatchedCentSweep) on the C1 shape of the paper's
centralized runs: n = 3, N = 5, the task-2 stop-and-go leader and spacing policy, T = 100 timesteps, initial states from
PlatoonEnv.reset of seeds 0..S-1.

Cases: 2-norm pwa_gear at S = 10, 256, 4096; 1-norm (MILP) at S = 10, 256; pwa_friction (discrete gears) at S = 256.
Per case one untimed full-size run, then the median of 3 timed runs; the largest difference between the runs' X shows
how far run-to-run scheduling moves the trajectories (ties between optimal leaves / vertices).  For S = 10 also 10
serial fleet_cent_mld.simulate() calls -- one seed after the other through the host-side agent loop, which is how the
paper's seeds run without the sweep.  The device name and power limit are read in the same run.
usage: python scripts/time_cent_sweep.py OUT_DIR   (writes OUT_DIR/time_cent_sweep.json)"""
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

n, N, T = 3, 5, 100
CASES = [("2-norm", "pwa_gear", True, 10), ("2-norm", "pwa_gear", True, 256), ("2-norm", "pwa_gear", True, 4096),
         ("1-norm", "pwa_gear", False, 10), ("1-norm", "pwa_gear", False, 256), ("friction", "pwa_friction", True, 256)]


def device_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def sim_for(model, quadratic):
    sim = hvp.Sim_n_task_2(n, seed=0, N=N)
    sim.vehicle_model_type, sim.quadratic_cost, sim.ep_len = model, quadratic, T
    return sim


def initial_states(sim, S):
    env, _, _, _ = make_env_and_systems(sim, forward_quadratic=True)
    return np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                                dtype=np.float64).reshape(-1) for s in range(S)])


def timed(sim, ctx, x0, lx):
    sw = SW.BatchedCentSweep(n, N, masses=sim.masses, spacing_policy=sim.spacing_policy, quadratic_cost=sim.quadratic_cost,
                             model=sim.vehicle_model_type, ctx=ctx)
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = sw.run(x0, lx, T)            # ends with a device synchronise and the read-back
        return time.perf_counter() - t0, r
    finally:
        sw.close()


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    out = sys.argv[1]
    os.makedirs(out, exist_ok=True)
    ctx = hvp.Context(0)
    res = dict(device=device_info(), workload=dict(n=n, N=N, T=T, leader="task-2 stop-and-go", policy="ConstantTimePolicy(10, 3)"),
               cases=[])
    print(res["device"], flush=True)
    for norm, model, quadratic, S in CASES:
        sim = sim_for(model, quadratic)
        lx = sim.leader_trajectory.get_leader_trajectory()
        x0 = initial_states(sim, S)
        timed(sim, ctx, x0, lx)           # full-size warm-up
        times, outs = [], []
        for _ in range(3):
            dt, r = timed(sim, ctx, x0, lx)
            times.append(dt)
            outs.append(r)
        med = float(np.median(times))
        r = outs[-1]
        st, cnt = np.unique(r["status"], return_counts=True)
        row = dict(norm=norm, model=model, S=S, times_s=times, median_s=med, scenario_timesteps_per_s=S * T / med,
                   solves_per_s=S * T / med, mean_nodes=float(r["nodes"].mean()),
                   status_counts={int(a): int(b) for a, b in zip(st, cnt)}, rollout_errors=int((r["errors"] != 0).sum()),
                   max_dX_between_runs=float(max(np.nanmax(np.abs(o["X"] - r["X"])) for o in outs[:-1])))
        if S == 10:
            hvp.fleet_cent_mld.simulate(sim, seed=0, ep_len=T)                  # warm-up of the host path
            t0 = time.perf_counter()
            for s in range(S):
                hvp.fleet_cent_mld.simulate(sim, seed=s, ep_len=T)
            dt = time.perf_counter() - t0
            row["serial_simulate"] = dict(calls=S, total_s=dt, scenario_timesteps_per_s=S * T / dt)
        res["cases"].append(row)
        print(json.dumps(row), flush=True)
    with open(os.path.join(out, "time_cent_sweep.json"), "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
