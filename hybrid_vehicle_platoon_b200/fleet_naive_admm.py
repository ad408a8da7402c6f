"""Drop-in for the reference's fleet_naive_admm.py (config 3): non-convex ADMM over per-vehicle MIQPs with
free copies of the neighbours' states.  LocalMpcADMM solves on the GPU; ADMMCoordinator follows
fleet_naive_admm.py:320-587 with the n independent x-updates of a round batched into one launch per
distinct formulation."""
from __future__ import annotations

import numpy as np

from ._sim import collect, make_env_and_systems, save_results
from .agents import MldAgent
from .misc import Params, Sim
from .mpc import LocalMpcADMM, solve_compiled_batch

LocalMpcGear = LocalMpcADMM       # the model type of the system dict selects the gear formulation


class ADMMCoordinator(MldAgent):
    def __init__(self, leader_index: int, local_mpcs, admm_iters: int, ep_len: int, N: int, leader_x: np.ndarray,
                 ts: float, rho: float) -> None:
        super().__init__(local_mpcs[0])
        self.n, self.leader_index = len(local_mpcs), leader_index
        self.agents = [MldAgent(m) for m in local_mpcs]
        self.leader_x, self.nx_l, self.nu_l = leader_x, 2, 1
        self.ep_len, self.ts, self.N, self.admm_iters, self.rho = ep_len, ts, N, admm_iters, rho
        self.y_front_list = [np.zeros((2, N + 1)) for _ in range(self.n)]
        self.y_back_list = [np.zeros((2, N + 1)) for _ in range(self.n)]
        self.z_list = [np.zeros((2, N + 1)) for _ in range(self.n)]
        self.solve_times = np.zeros((ep_len, 1))
        self.node_counts = np.zeros((ep_len, 1))
        self.temp_solve_time = 0
        self.temp_node_count = 0

    def get_control(self, state):
        n, ag = self.n, self.agents
        state = np.asarray(state, dtype=np.float64)
        xl = [state[2 * i:2 * (i + 1), :] for i in range(n)]
        # initial guess for the coupling variables: previous solutions, shifted (:392-402)
        for i in range(n):
            if i != 0:
                xa = ag[i - 1].get_predicted_state(shifted=True)
                if xa is not None:
                    ag[i].mpc.set_front_vars(self.y_front_list[i], xa)
            if i != n - 1:
                xb = ag[i + 1].get_predicted_state(shifted=True)
                if xb is not None:
                    ag[i].mpc.set_back_vars(self.y_back_list[i], xb)
        u = [None] * n
        for _ in range(self.admm_iters):
            # x-update: n independent local MIQPs (:407-411)
            res = solve_compiled_batch([a.mpc for a in ag], xl)
            for i, (a, (ui, info)) in enumerate(zip(ag, res)):
                a._store(info)
                u[i] = ui
            # z-update and y-update together (:421-447)
            for i in range(n):
                if n == 1:
                    self.z_list[i] = ag[i].mpc.x.X.copy()
                elif i == 0:
                    self.z_list[i] = (1.0 / 2.0) * (ag[i].mpc.x.X + ag[i + 1].mpc.x_front.X)
                    self.y_front_list[i + 1] += self.rho * (ag[i + 1].mpc.x_front.X - self.z_list[i])
                elif i == n - 1:
                    self.z_list[i] = (1.0 / 2.0) * (ag[i].mpc.x.X + ag[i - 1].mpc.x_back.X)
                    self.y_back_list[i - 1] += self.rho * (ag[i - 1].mpc.x_back.X - self.z_list[i])
                else:
                    self.z_list[i] = (1.0 / 3.0) * (ag[i].mpc.x.X + ag[i + 1].mpc.x_front.X + ag[i - 1].mpc.x_back.X)
                    self.y_front_list[i + 1] += self.rho * (ag[i + 1].mpc.x_front.X - self.z_list[i])
                    self.y_back_list[i - 1] += self.rho * (ag[i - 1].mpc.x_back.X - self.z_list[i])
            # push (y, z) back into the local models (:453-468)
            for i in range(n):
                if i != 0:
                    ag[i].mpc.set_front_vars(self.y_front_list[i], self.z_list[i - 1])
                if i != n - 1:
                    ag[i].mpc.set_back_vars(self.y_back_list[i], self.z_list[i + 1])
            self.temp_solve_time += max(a.run_time for a in ag)
            self.temp_node_count = max(max(a.node_count for a in ag), self.temp_node_count)
        if u[0].shape[0] > self.nu_l:          # [u ; gears] per vehicle -> all throttles, then all gears (:556-564)
            return np.vstack((np.vstack([ui[:self.nu_l, :] for ui in u]), np.vstack([ui[self.nu_l:, :] for ui in u]))), {}
        return np.vstack(u), {}

    def on_timestep_end(self, env, episode: int, timestep: int) -> None:
        self.agents[self.leader_index].mpc.set_leader_x(self.leader_x[:, timestep:timestep + self.N + 1])
        self.solve_times[env.step_counter - 1, :] = self.temp_solve_time
        self.node_counts[env.step_counter - 1, :] = self.temp_node_count
        self.temp_solve_time = 0
        self.temp_node_count = 0

    def on_episode_start(self, env, episode: int, state) -> None:
        self.agents[self.leader_index].mpc.set_leader_x(self.leader_x[:, 0:self.N + 1])


def simulate(sim: Sim, admm_iters: int = 20, save: bool = False, plot: bool = False, seed: int = 1,
             thread_limit=None, leader_index: int = 0, ep_len=None, env_class=None):
    """fleet_naive_admm.simulate (:590-696)."""
    n, N, ts = sim.n, sim.N, Params.ts
    leader_x = sim.leader_trajectory.get_leader_trajectory()
    env, platoon, systems, ep_len = make_env_and_systems(sim, leader_index, ep_len, env_class)
    mpcs = [LocalMpcADMM(N, systems[i], rho=0.5, spacing_policy=sim.spacing_policy, is_front=(i == 0),
                         is_leader=(i == leader_index), is_trailer=(i == n - 1), thread_limit=thread_limit)
            for i in range(n)]
    agent = ADMMCoordinator(leader_index=leader_index, local_mpcs=mpcs, admm_iters=admm_iters, rho=0.5,
                            ep_len=ep_len, N=N, leader_x=leader_x, ts=ts)
    agent.evaluate(env=env, episodes=1, seed=seed)
    return collect(env, agent, leader_x, f"admm_{admm_iters}_{sim.id}_seed_{seed}.pkl", save)


def simulate_many(sim: Sim, seeds, admm_iters: int = 20, leader_index: int = 0, ep_len=None, save: bool = False,
                  strict: bool = True, ctx=None):
    """simulate() for several seeds of one configuration in ONE on-device closed loop (sweep.BatchedAdmmSweep): the
    paper's "10 seeds of a configuration" in one call.  Each seed's initial state is PlatoonEnv.reset with the seed
    MldAgent.evaluate derives from it, the masses and d_safe are the env's, rho is 0.5 and the solver options are the
    ones simulate() would use (mpc.OPTIONS); sim.real_vehicle_as_reference goes to the rollout as simulate() gives it to
    PlatoonEnv.  Every Sim simulate() accepts is accepted (this controller ignores open_loop and quadratic_cost), except
    n < 2: the batched loop needs at least two vehicles.  Returns one dict per seed with simulate()'s 7 objects and
    shapes, except solve_times, which is NaN: a batched launch has no per-scenario solve time; node_counts is the
    largest node count over the rounds and vehicles of a timestep.  save=True writes simulate()'s pickle per seed.
    strict=True raises what simulate() would after the run, naming the seed and timestep: RuntimeError("Infeasible
    problem encountered ...") for a solve that was not optimal (RuntimeWarning with pwa_friction, as the gear MPC
    raises), the rollout's error otherwise, whichever comes first in the episode; strict=False returns the episodes as
    computed, with a vehicle whose solve was not optimal applying zero input (gear 6), as solve_mpc(raises=False)."""
    from .env import raise_rollout_error
    from .mpc import OPTIONS
    from .sweep import BatchedAdmmSweep
    n, N = sim.n, sim.N
    if n < 2:
        raise ValueError("the batched ADMM loop needs at least two vehicles")
    seeds = [int(s) for s in seeds]
    leader_x = sim.leader_trajectory.get_leader_trajectory()
    env, _, _, ep_len = make_env_and_systems(sim, leader_index, ep_len, None)
    base = env.unwrapped
    x0 = np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                              dtype=np.float64).reshape(2 * n) for s in seeds])
    sw = BatchedAdmmSweep(n, N, admm_iters=admm_iters, rho=0.5, masses=base.masses, spacing_policy=sim.spacing_policy,
                          leader_index=leader_index, d_safe=base.d_safe, model=sim.vehicle_model_type,
                          mip_gap=OPTIONS.mip_gap, time_limit_ms=OPTIONS.time_limit * 1e3,
                          real_vehicle_as_reference=sim.real_vehicle_as_reference, ctx=ctx)
    try:
        r = sw.run(x0, leader_x, ep_len)
    finally:
        sw.close()
    if strict:
        # what simulate() meets first in each episode; the first episode (in seed order) that meets one is reported
        for j, seed in enumerate(seeds):
            bad_t, _, st = (int(v) for v in r["failed_at"][j])
            err_t = np.nonzero(r["errors"][:, j])[0]
            if bad_t >= 0 and (not err_t.size or bad_t <= err_t[0]):
                if sim.vehicle_model_type == "pwa_friction":      # mpcs/mpc_gear.py:127-128
                    raise RuntimeWarning(f"gear mpc is infeasible (status {st}; seed {seed}, timestep {bad_t})")
                raise RuntimeError(f"Infeasible problem encountered (status {st}). (seed {seed}, timestep {bad_t})")
            if err_t.size:
                try:
                    raise_rollout_error(int(r["errors"][err_t[0], j]))
                except RuntimeError as e:
                    raise RuntimeError(f"{e} (seed {seed}, timestep {int(err_t[0])})") from None
    out = []
    for j, seed in enumerate(seeds):
        # shapes of collect(): X (T+1,2n), U (T,n|2n), R (T,1,1), solve_times / node_counts (T,1), violations (T,)
        res = dict(X=r["X"][:, j].copy(), U=r["U"][:, j].copy(), R=r["R"][:, j].reshape(ep_len, 1, 1).copy(),
                   solve_times=np.full((ep_len, 1), np.nan), node_counts=r["nodes"][:, j].astype(np.float64).reshape(ep_len, 1),
                   violations=np.where(r["violations"][:, j] != 0, 100.0, 0.0), leader_x=leader_x)
        if save:
            save_results(res, f"admm_{admm_iters}_{sim.id}_seed_{seed}.pkl")
        out.append(res)
    return out
