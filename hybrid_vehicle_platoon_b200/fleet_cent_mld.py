"""Drop-in for the reference's fleet_cent_mld.py: centralized MLD MPC of the whole platoon (config 1).
MpcMldCent / MpcGearCent solve on the GPU (compiled-MPC kernel); TrackingCentralizedAgent and simulate()
follow fleet_cent_mld.py:80-213."""
from __future__ import annotations

import numpy as np

from ._sim import collect, make_env_and_systems, save_results
from .agents import MldAgent
from .misc import Params, Sim
from .mpc import MpcGearCent, MpcMldCent  # noqa: F401


class TrackingCentralizedAgent(MldAgent):
    def __init__(self, mpc: MpcMldCent, ep_len: int, N: int, leader_x: np.ndarray) -> None:
        self.solve_times = np.zeros((ep_len, 1))
        self.node_counts = np.zeros((ep_len, 1))
        self.bin_var_counts = np.zeros((ep_len, 1))
        self.N, self.leader_x = N, leader_x
        super().__init__(mpc)

    def on_timestep_end(self, env, episode: int, timestep: int) -> None:
        # time step starts from 1, so this sets the cost accurately for the next time-step
        self.mpc.set_leader_traj(self.leader_x[:, timestep:(timestep + self.N + 1)])
        self.solve_times[env.step_counter - 1, :] = self.run_time
        self.node_counts[env.step_counter - 1, :] = self.node_count
        self.bin_var_counts[env.step_counter - 1, :] = self.num_bin_vars
        return super().on_timestep_end(env, episode, timestep)

    def on_episode_start(self, env, episode: int, state) -> None:
        self.mpc.set_leader_traj(self.leader_x[:, 0:self.N + 1])
        return super().on_episode_start(env, episode, state)


def simulate(sim: Sim, save: bool = False, plot: bool = False, seed: int = 1, thread_limit=None,
             leader_index: int = 0, ep_len=None, env_class=None):
    """fleet_cent_mld.simulate (:104-213); returns the 7 result objects as a dict."""
    n, N = sim.n, sim.N
    leader_x = sim.leader_trajectory.get_leader_trajectory()
    env, platoon, systems, ep_len = make_env_and_systems(sim, leader_index, ep_len, env_class,
                                                         forward_quadratic=True)
    if sim.vehicle_model_type not in ("pwa_gear", "pwa_friction"):
        raise NotImplementedError(f"{sim.vehicle_model_type}: the non-convex nonlinear MPC is not built (SURVEY 8f)")
    mpc = MpcMldCent(n, N, systems, spacing_policy=sim.spacing_policy, leader_index=leader_index,
                     quadratic_cost=sim.quadratic_cost, thread_limit=thread_limit,
                     real_vehicle_as_reference=sim.real_vehicle_as_reference)
    agent = TrackingCentralizedAgent(mpc, ep_len, N, leader_x)
    agent.evaluate(env=env, episodes=1, seed=seed, open_loop=sim.open_loop)
    return collect(env, agent, leader_x, f"cent_{sim.id}_seed_{seed}.pkl", save)


def simulate_many(sim: Sim, seeds, leader_index: int = 0, ep_len=None, save: bool = False, strict: bool = True, ctx=None):
    """simulate() for several seeds of one configuration in ONE on-device closed loop (sweep.BatchedCentSweep): the
    paper's "10 seeds of a configuration" in one call.  Each seed's initial state is PlatoonEnv.reset with the seed
    MldAgent.evaluate derives from it, the solver options are the ones simulate() would use (mpc.OPTIONS).  Returns one
    dict per seed with simulate()'s 7 objects and shapes, except solve_times, which is NaN: a batched launch has no
    per-scenario solve time.  save=True writes simulate()'s pickle per seed.  strict=True raises what simulate() would
    (RuntimeError; RuntimeWarning for the discrete-gear MPC, mpcs/mpc_gear.py:127-128) after the run if any solve was
    not optimal or the rollout failed; strict=False returns the episodes with zero inputs (gear 6) where a solve failed."""
    from .env import raise_rollout_error
    from .mpc import OPTIONS
    from .sweep import BatchedCentSweep
    if sim.open_loop or sim.real_vehicle_as_reference:
        raise NotImplementedError("simulate_many runs closed loops with the leader trajectory as reference only")
    if sim.vehicle_model_type not in ("pwa_gear", "pwa_friction"):
        raise NotImplementedError(f"{sim.vehicle_model_type}: the non-convex nonlinear MPC is not built (SURVEY 8f)")
    n, N = sim.n, sim.N
    seeds = [int(s) for s in seeds]
    leader_x = sim.leader_trajectory.get_leader_trajectory()
    env, _, _, ep_len = make_env_and_systems(sim, leader_index, ep_len, None, forward_quadratic=True)
    base = env.unwrapped
    x0 = np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                              dtype=np.float64).reshape(2 * n) for s in seeds])
    sw = BatchedCentSweep(n, N, masses=base.masses, spacing_policy=sim.spacing_policy, leader_index=leader_index,
                          quadratic_cost=sim.quadratic_cost, model=sim.vehicle_model_type, d_safe=base.d_safe,
                          mip_gap=OPTIONS.mip_gap, time_limit_ms=OPTIONS.time_limit * 1e3, ctx=ctx)
    try:
        r = sw.run(x0, leader_x, ep_len)
    finally:
        sw.close()
    if strict:
        bad = r["status"] != 2
        if bad.any():
            t, j = (int(v) for v in np.argwhere(bad)[0])
            if sim.vehicle_model_type == "pwa_friction":
                raise RuntimeWarning(f"gear mpc for state {r['X'][t, j]} is infeasible (seed {seeds[j]}, timestep {t}).")
            raise RuntimeError(f"Infeasible problem encountered (status {int(r['status'][t, j])}; seed {seeds[j]}, "
                               f"timestep {t}).")
        if r["errors"].any():
            raise_rollout_error(int(r["errors"][np.nonzero(r["errors"])][0]))
    out = []
    for j, seed in enumerate(seeds):
        # shapes of collect(): X (T+1,2n), U (T,n|2n), R (T,1,1), solve_times / node_counts (T,1), violations (T,)
        res = dict(X=r["X"][:, j].copy(), U=r["U"][:, j].copy(), R=r["R"][:, j].reshape(ep_len, 1, 1).copy(),
                   solve_times=np.full((ep_len, 1), np.nan), node_counts=r["nodes"][:, j].astype(np.float64).reshape(ep_len, 1),
                   violations=np.where(r["violations"][:, j] != 0, 100.0, 0.0), leader_x=leader_x)
        if save:
            save_results(res, f"cent_{sim.id}_seed_{seed}.pkl")
        out.append(res)
    return out
