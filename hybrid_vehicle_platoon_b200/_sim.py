"""Shared scaffolding of the fleet scripts' simulate() functions (env + wrappers + result schema)."""
from __future__ import annotations

import pickle

import numpy as np

from .agents import MonitorEpisodes, TimeLimit
from .misc import Params


def make_env_and_systems(sim, leader_index: int = 0, ep_len=None, env_class=None, forward_real_ref=True,
                         forward_quadratic=False):
    from .env import PlatoonEnv
    from .models import Platoon
    env_class = env_class or PlatoonEnv
    ep_len = ep_len or sim.ep_len
    platoon = Platoon(sim.n, vehicle_type=sim.vehicle_model_type, masses=sim.masses)
    systems = platoon.get_vehicle_system_dicts(Params.ts)
    kw = {}
    if forward_real_ref:
        kw["real_vehicle_as_reference"] = sim.real_vehicle_as_reference
    if forward_quadratic:
        kw["quadratic_cost"] = sim.quadratic_cost
    env = MonitorEpisodes(TimeLimit(env_class(
        n=sim.n, platoon=platoon, leader_trajectory=sim.leader_trajectory, spacing_policy=sim.spacing_policy,
        start_from_platoon=sim.start_from_platoon, ep_len=ep_len, leader_index=leader_index, **kw),
        max_episode_steps=ep_len))
    return env, platoon, systems, ep_len


def collect(env, agent, leader_x, fname: str, save: bool, node_counts=None):
    """The reference's 7 result objects (e.g. fleet_cent_mld.py:185-213): X (T+1,2n), U (T,n|2n), R (T,1,1),
    solve_times (T,1), node_counts (T,1), violations (T,), leader_x (2,T+50)."""
    X, U, R = env.observations[0].squeeze(), env.actions[0].squeeze(), env.rewards[0]
    out = dict(X=X, U=U, R=R, solve_times=np.asarray(agent.solve_times),
               node_counts=agent.node_counts if node_counts is None else node_counts,
               violations=env.unwrapped.viol_counter[-1], leader_x=leader_x)
    if save:
        save_results(out, fname)
    return out


def save_results(out: dict, fname: str) -> None:
    """The reference's pickle: the 7 result objects dumped one after the other, in this order."""
    with open(fname, "wb") as f:
        for k in ("X", "U", "R", "solve_times", "node_counts", "violations", "leader_x"):
            pickle.dump(out[k], f)
