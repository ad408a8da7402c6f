"""Drop-in for the reference's fleet_event_based.py: each agent optimises itself and up to one neighbour
each side, the agent with the largest cost decrease (> threshold) wins an iteration.  LocalMpc solves and
eval_cost run on the GPU, batched over the agents of an iteration; TrackingEventBasedCoordinator follows
fleet_event_based.py:413-646."""
from __future__ import annotations

import numpy as np

from ._sim import collect, make_env_and_systems, save_results
from .agents import MldAgent
from .misc import Params, Sim
from .mpc import EventLocalMpc as LocalMpc, eval_compiled_batch, solve_compiled_batch

LocalMpcGear = LocalMpc
threshold = 10  # cost improvement must be more than this to consider communication (fleet_event_based.py:23)


class TrackingEventBasedCoordinator(MldAgent):
    def __init__(self, local_mpcs, vehicles, ep_len: int, N: int, leader_x: np.ndarray, discrete_gears: bool,
                 ts: float, event_iters: int = 4, leader_index: int = 0) -> None:
        super().__init__(local_mpcs[0])
        self.n = len(local_mpcs)
        self.agents = [MldAgent(m) for m in local_mpcs]
        self.nx_l, self.nu_l = 2, 1
        self.vehicles, self.num_iters, self.leader_x, self.ts, self.N = vehicles, event_iters, leader_x, ts, N
        self.discrete_gears, self.leader_index = discrete_gears, leader_index
        self.state_guesses = [np.zeros((2, N + 1)) for _ in range(self.n)]
        self.control_guesses = [np.zeros((1, N)) for _ in range(self.n)]
        self.gear_guesses = [np.zeros((1, N)) for _ in range(self.n)]
        self.solve_times = np.zeros((ep_len, 1))
        self.node_counts = np.zeros((ep_len, 1))
        self.temp_solve_time = 0
        self.temp_node_count = 0

    def _members(self, i):
        if i == 0:
            return [0, 1]
        if i == self.n - 1:
            return [self.n - 2, self.n - 1]
        return [i - 1, i, i + 1]

    def get_control(self, state):
        n, ag = self.n, self.agents
        state = np.asarray(state, dtype=np.float64)
        temp_costs = [None] * n
        for _ in range(self.num_iters):
            best_cost_dec, best_idx = -float("inf"), -1
            x_ls, xg, ug = [], [], []
            for i in range(n):
                mem = self._members(i)
                x_ls.append(np.vstack([state[2 * j:2 * (j + 1), :] for j in mem]))
                xg.append(np.vstack([self.state_guesses[j] for j in mem]))
                ug.append(np.vstack([self.control_guesses[j] for j in mem]))
                # constant predictions for the neighbours of neighbours (:504-508)
                if i > 1:
                    ag[i].mpc.set_x_f2(self.state_guesses[i - 2])
                if i < n - 2:
                    ag[i].mpc.set_x_b2(self.state_guesses[i + 2])
            # within one iteration the n evaluations and the n local MIQPs are independent (:470-521)
            costs = eval_compiled_batch([a.mpc for a in ag], xg, ug)
            res = solve_compiled_batch([a.mpc for a in ag], x_ls, raises=False)
            feasible_sol_flag = False
            for i in range(n):
                temp_costs[i] = float(costs[i])
                ag[i]._store(res[i][1])
                new_cost = ag[i].get_predicted_cost()
                if new_cost < float("inf"):
                    feasible_sol_flag = True
                if (temp_costs[i] - new_cost > best_cost_dec) and (temp_costs[i] - new_cost > threshold):
                    best_cost_dec, best_idx = temp_costs[i] - new_cost, i
            if not feasible_sol_flag:
                raise RuntimeWarning("No feasible solution found for any event based agent.")
            self.temp_solve_time += max(a.run_time for a in ag)
            self.temp_node_count = max(max(a.node_count for a in ag), self.temp_node_count)
            if best_idx < 0:                   # nobody improved: stop iterating (:568-569)
                break
            best_x, best_u = ag[best_idx].x_pred, ag[best_idx].u_pred
            for l, j in enumerate(self._members(best_idx)):     # the winner's plan overwrites the shared guesses
                self.state_guesses[j] = best_x[2 * l:2 * l + 2, :]
                self.control_guesses[j] = best_u[[l], :]
                if self.discrete_gears:
                    self.gear_guesses[j] = ag[best_idx].mpc.gears_pred[[l], :]
        u0 = np.vstack([self.control_guesses[i][:, [0]] for i in range(n)])
        if self.discrete_gears:
            return np.vstack((u0, np.vstack([self.gear_guesses[i][:, [0]] for i in range(n)]))), {}
        return u0, {}

    def _set_leader(self, leader_x):
        li = self.leader_index
        self.agents[li].mpc.set_leader_x(leader_x)
        if li > 0:
            self.agents[li - 1].mpc.set_leader_x(leader_x)
        if li < self.n - 1:
            self.agents[li + 1].mpc.set_leader_x(leader_x)

    def on_timestep_end(self, env, episode: int, timestep: int) -> None:
        self._set_leader(self.leader_x[:, timestep:timestep + self.N + 1])
        sh = lambda a: np.concatenate((a[:, 1:], a[:, -1:]), axis=1)     # shifted previous solution (:591-603)
        for i in range(self.n):
            self.state_guesses[i] = sh(self.state_guesses[i])
            self.control_guesses[i] = sh(self.control_guesses[i])
            if self.discrete_gears:
                self.gear_guesses[i] = sh(self.gear_guesses[i])
        self.solve_times[env.step_counter - 1, :] = self.temp_solve_time
        self.node_counts[env.step_counter - 1, :] = self.temp_node_count
        self.temp_solve_time = 0
        self.temp_node_count = 0

    def on_episode_start(self, env, episode: int, state) -> None:
        self._set_leader(self.leader_x[:, 0:self.N + 1])
        for i in range(self.n):                # first guesses: constant velocity (:620-634)
            xl = env.x[2 * i:2 * (i + 1), :]
            self.state_guesses[i] = self.extrapolate_position(xl[0, :], xl[1, :])
            if not self.discrete_gears:
                self.control_guesses[i] = self.vehicles[i].get_u_for_constant_vel(xl[1, 0]) * np.ones((1, self.N))
            else:
                j = self.vehicles[i].get_gear_from_velocity(xl[1, 0])
                self.gear_guesses[i] = j * np.ones((1, self.N))
                self.control_guesses[i] = self.vehicles[i].get_u_for_constant_vel(xl[1, 0], j) * np.ones((1, self.N))

    def extrapolate_position(self, initial_pos, initial_vel):
        x_pred = np.zeros((2, self.N + 1))
        x_pred[0, [0]] = initial_pos
        x_pred[1, [0]] = initial_vel
        for k in range(self.N):
            x_pred[0, [k + 1]] = x_pred[0, [k]] + self.ts * x_pred[1, [k]]
            x_pred[1, [k + 1]] = x_pred[1, [k]]
        return x_pred


def simulate(sim: Sim, event_iters: int = 4, save: bool = False, plot: bool = False, seed: int = 2,
             thread_limit=None, leader_index: int = 0, ep_len=None, env_class=None):
    """fleet_event_based.simulate (:649-767)."""
    n, N, ts = sim.n, sim.N, Params.ts
    if n < 2:
        raise ValueError("the event-based scheme needs at least two vehicles")
    leader_x = sim.leader_trajectory.get_leader_trajectory()
    env, platoon, systems, ep_len = make_env_and_systems(sim, leader_index, ep_len, env_class, forward_real_ref=False)
    discrete_gears = sim.vehicle_model_type == "pwa_friction"
    mpcs = [LocalMpc(N, systems=(systems[:2] if i == 0 else (systems[-2:] if i == n - 1 else systems[i - 1:i + 2])),
                     num_vehicles_in_front=i if i < 2 else 2,
                     num_vehicles_behind=(n - 1) - i if i > n - 3 else 2,
                     rel_leader_index=(-1 if i == leader_index - 1 else (0 if i == leader_index else
                                                                         (1 if i == leader_index + 1 else None))),
                     spacing_policy=sim.spacing_policy, thread_limit=thread_limit)
            for i in range(n)]
    agent = TrackingEventBasedCoordinator(mpcs, vehicles=platoon.get_vehicles(), ep_len=ep_len, N=N, leader_x=leader_x,
                                          discrete_gears=discrete_gears, ts=ts, event_iters=event_iters,
                                          leader_index=leader_index)
    agent.evaluate(env=env, episodes=1, seed=seed)
    return collect(env, agent, leader_x, f"event_{event_iters}_{sim.id}_seed_{seed}.pkl", save)


def simulate_many(sim: Sim, seeds, event_iters: int = 4, leader_index: int = 0, ep_len=None, save: bool = False,
                  strict: bool = True, ctx=None):
    """simulate() for several seeds of one configuration in ONE on-device closed loop (sweep.BatchedEventSweep): the
    paper's "10 seeds of a configuration" in one call.  Each seed's initial state is PlatoonEnv.reset with the seed
    MldAgent.evaluate derives from it, the masses are the env's and the solver options are the ones simulate() would use
    (mpc.OPTIONS).  Returns one dict per seed with simulate()'s 7 objects and shapes, except solve_times, which is NaN: a
    batched launch has no per-scenario solve time; node_counts is the largest node count over the iterations and agents
    of a timestep.  save=True writes simulate()'s pickle per seed.  strict=True raises what simulate() would after the
    run, naming the seed and timestep: RuntimeWarning for an iteration in which no agent's MIQP was solved, the rollout's
    error otherwise; strict=False returns the episodes as computed."""
    from .env import raise_rollout_error
    from .mpc import OPTIONS
    from .sweep import BatchedEventSweep
    n, N = sim.n, sim.N
    if n < 2:
        raise ValueError("the event-based scheme needs at least two vehicles")
    seeds = [int(s) for s in seeds]
    leader_x = sim.leader_trajectory.get_leader_trajectory()
    env, _, _, ep_len = make_env_and_systems(sim, leader_index, ep_len, None, forward_real_ref=False)
    base = env.unwrapped
    x0 = np.stack([np.asarray(env.reset(seed=int(np.random.SeedSequence(s).generate_state(1)[0]))[0],
                              dtype=np.float64).reshape(2 * n) for s in seeds])
    sw = BatchedEventSweep(n, N, event_iters=event_iters, masses=base.masses, spacing_policy=sim.spacing_policy,
                           leader_index=leader_index, d_safe=base.d_safe, threshold=threshold, model=sim.vehicle_model_type,
                           mip_gap=OPTIONS.mip_gap, time_limit_ms=OPTIONS.time_limit * 1e3, ctx=ctx)
    try:
        r = sw.run(x0, leader_x, ep_len)
    finally:
        sw.close()
    if strict:
        # what simulate() meets first in each episode; the first episode (in seed order) that meets one is reported
        for j, seed in enumerate(seeds):
            bad_t = np.nonzero(~r["feasible"][:, j])[0]
            err_t = np.nonzero(r["errors"][:, j])[0]
            if bad_t.size and (not err_t.size or bad_t[0] <= err_t[0]):
                raise RuntimeWarning(f"No feasible solution found for any event based agent. (seed {seed}, timestep "
                                     f"{int(bad_t[0])})")
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
            save_results(res, f"event_{event_iters}_{sim.id}_seed_{seed}.pkl")
        out.append(res)
    return out
