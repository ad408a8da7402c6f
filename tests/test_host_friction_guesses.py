"""The vectorised first guesses of the event-based sweep with discrete gears (sweep.friction_gear_from_velocity,
sweep.friction_const_vel_u) against PwaFrictionVehicle's scalar methods, bit for bit, on the CPU."""
import warnings

import numpy as np
import torch

from hybrid_vehicle_platoon_b200.models import PwaFrictionVehicle, Vehicle
from hybrid_vehicle_platoon_b200.sweep import friction_const_vel_u, friction_gear_from_velocity


def _velocities():
    """A grid over and beyond the velocity range, every gear-window edge and its neighbouring doubles, the friction
    region edge alpha, and the integer speeds PlatoonEnv.reset draws (5..34 m/s)."""
    edges = sorted(set(Vehicle.vl + Vehicle.vh + [PwaFrictionVehicle.alpha]))
    near = [np.nextafter(e, d) for e in edges for d in (-np.inf, np.inf)]
    v = np.concatenate([np.linspace(0.0, 60.0, 2401), near, np.arange(5.0, 35.0), [-3.0, 100.0]])
    return np.array([x for x in v if x not in (Vehicle.v_min, Vehicle.v_max)])   # the scalar method raises there


def test_gear_from_velocity_matches_scalar():
    v = _velocities()
    veh = PwaFrictionVehicle(800.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = np.array([veh.get_gear_from_velocity(float(x)) for x in v])
    got = friction_gear_from_velocity(torch.as_tensor(v)).numpy()
    np.testing.assert_array_equal(got, ref)
    assert (got[v < Vehicle.v_min] == 1).all() and (got[v > Vehicle.v_max] == 6).all()
    # the two speeds that no open gear window contains: the scalar method raises, the vectorised one returns 0
    assert friction_gear_from_velocity(torch.tensor([Vehicle.v_min, Vehicle.v_max], dtype=torch.float64)).tolist() == [0, 0]


def test_const_vel_throttle_matches_scalar():
    v = _velocities()
    gear = friction_gear_from_velocity(torch.as_tensor(v))
    for m in (800.0, 650.0, 1137.25):
        veh = PwaFrictionVehicle(m)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = np.array([veh.get_u_for_constant_vel(float(x), int(j)) for x, j in zip(v, gear.tolist())])
        got = friction_const_vel_u(torch.as_tensor(v), gear, torch.full((len(v),), m, dtype=torch.float64)).numpy()
        np.testing.assert_array_equal(got, ref, err_msg=f"m={m}")
    # per-element masses in a (S, n) layout, as the sweep calls it
    rng = np.random.default_rng(3)
    vv = rng.choice(v, (16, 5))
    mm = rng.uniform(600.0, 1200.0, (16, 5))
    gg = friction_gear_from_velocity(torch.as_tensor(vv))
    got = friction_const_vel_u(torch.as_tensor(vv), gg, torch.as_tensor(mm)).numpy()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = np.array([[PwaFrictionVehicle(mm[s, i]).get_u_for_constant_vel(float(vv[s, i]), int(gg[s, i]))
                         for i in range(5)] for s in range(16)])
    np.testing.assert_array_equal(got, ref)
