"""Wall clock of the naive-ADMM on-device closed loop (sweep.BatchedAdmmSweep / fleet_naive_admm.simulate_many).

Cases (initial states from PlatoonEnv.reset of seeds 0..S-1, as simulate_many takes them):
  * default Sim, n = 3, N = 5, admm_iters = 10, T = 30: simulate_many of 10 seeds against 10 serial
    fleet_naive_admm.simulate() calls, and the sweep at S = 256 and 1024;
  * the C3 shape, Sim_n_task_2(15, N = 8), admm_iters = 20, task-2 stop-and-go leader, T = 4, S = 10 and 1024;
  * pwa_friction (discrete gears), n = 3, N = 3, admm_iters = 4, T = 10, S = 256.
Every sweep case runs two arms, alternated: the roles' solves on forked streams (fork, the default) and in sequence.
Per arm one untimed full-size run, then the median of 3 timed runs.  Each record gives the episode time,
scenario-timesteps and scenario-rounds per second, the fraction of optimal solves, the mean node count and the largest
|dX| against the first arm.  The device name, power limit and max SM clock are read in the same run.
usage: python scripts/time_admm_sweep.py OUT_DIR   (writes OUT_DIR/time_admm_sweep.json)"""
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

ARMS = {"fork": dict(fork=True), "no_fork": dict(fork=False)}


def device_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def default_sim(n, N, model="pwa_gear"):
    sim = hvp.Sim()
    sim.n, sim.N, sim.vehicle_model_type = n, N, model
    sim.id = f"default_n_{n}_N_{N}"
    return sim


# (label, sim factory, admm_iters, T, batch sizes, serial simulate() comparison at S = 10)
CASES = [("default", lambda: default_sim(3, 5), 10, 30, (10, 256, 1024), True),
         ("C3", lambda: hvp.Sim_n_task_2(15, seed=7, N=8), 20, 4, (10, 1024), False),
         ("friction", lambda: default_sim(3, 3, "pwa_friction"), 4, 10, (256,), False)]


def initial_states(sim, S):
    env, _, _, _ = make_env_and_systems(sim)
    return np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                                dtype=np.float64).reshape(-1) for s in range(S)]), env.unwrapped.masses


def timed(sim, ctx, x0, masses, lx, T, iters, arm):
    sw = SW.BatchedAdmmSweep(sim.n, sim.N, admm_iters=iters, masses=masses, spacing_policy=sim.spacing_policy,
                             model=sim.vehicle_model_type, ctx=ctx, **ARMS[arm])
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
    res = dict(device=device_info(), cases=[])
    print(res["device"], flush=True)
    for label, make, iters, T, sizes, serial in CASES:
        sim = make()
        lx = sim.leader_trajectory.get_leader_trajectory()
        for S in sizes:
            x0, masses = initial_states(sim, S)
            for arm in ARMS:
                timed(sim, ctx, x0, masses, lx, T, iters, arm)      # full-size warm-up of every arm
            times = {a: [] for a in ARMS}
            outs = {}
            for _ in range(3):                                        # the arms alternate
                for arm in ARMS:
                    dt, r = timed(sim, ctx, x0, masses, lx, T, iters, arm)
                    times[arm].append(dt)
                    outs[arm] = r
            first = next(iter(ARMS))
            for arm in ARMS:
                med = float(np.median(times[arm]))
                r = outs[arm]
                row = dict(case=label, model=sim.vehicle_model_type, n=sim.n, N=sim.N, admm_iters=iters, T=T, S=S, arm=arm,
                           times_s=times[arm], median_s=med, scenario_timesteps_per_s=S * T / med,
                           scenario_rounds_per_s=S * T * iters / med, optimal_frac=float((r["status"] == 2).mean()),
                           failed_scenarios=int((r["failed_at"][:, 0] >= 0).sum()), mean_nodes=float(r["nodes"].mean()),
                           rollout_errors=int((r["errors"] != 0).sum()),
                           max_dX_vs_first=float(np.nanmax(np.abs(r["X"] - outs[first]["X"]))))
                res["cases"].append(row)
                print(json.dumps(row), flush=True)
            if serial and S == 10:
                seeds = list(range(S))
                hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=iters, ep_len=T, strict=False, ctx=ctx)  # warm-up
                many = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    hvp.fleet_naive_admm.simulate_many(sim, seeds, admm_iters=iters, ep_len=T, strict=False, ctx=ctx)
                    many.append(time.perf_counter() - t0)
                row = dict(case=label, n=sim.n, N=sim.N, admm_iters=iters, T=T, S=S, arm="simulate_many", times_s=many,
                           median_s=float(np.median(many)))
                try:
                    hvp.fleet_naive_admm.simulate(sim, admm_iters=iters, seed=0, ep_len=T)    # warm-up of the host path
                    t0 = time.perf_counter()
                    for s in seeds:
                        hvp.fleet_naive_admm.simulate(sim, admm_iters=iters, seed=s, ep_len=T)
                    dt = time.perf_counter() - t0
                    row.update(serial_simulate_s=dt, speedup=dt / row["median_s"])
                except (RuntimeError, RuntimeWarning) as e:    # simulate() raises where the sweep reports
                    row.update(serial_simulate_error=repr(e))
                res["cases"].append(row)
                print(json.dumps(row), flush=True)
            with open(os.path.join(out, "time_admm_sweep.json"), "w") as f:
                json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
