"""Scenario tables: per-env episode conditions that every reset applies in place of the random draws (`X500Task.set_scenarios`,
C ABI `ozl_set_scenarios`; row layout OZL_SCN_* in include/ouzelum_b200.h, `_lib.SCENARIO_LAYOUT`).

    rows = scenarios.fault_grid(env.num_envs, rotors=[0, 1, 2, 3], onsets=[0, 300], effectiveness=[0.1, 0.5])
    env.set_scenarios(rows)
    result = scenarios.evaluate(env, lambda obs: policy(obs["obs"]), steps=4000)

Two policies evaluated on the same table see the same faults, spawn poses and body parameters in every episode.
"""
import itertools

import torch

from ._lib import SCENARIO_LAYOUT, SCENARIO_WIDTH

_ROTOR, _ONSET, _EFF = (SCENARIO_LAYOUT[k] for k in ("OZL_SCN_FAULT_ROTOR", "OZL_SCN_FAULT_ONSET", "OZL_SCN_FAULT_EFF"))


def empty(n):
    """[n, SCENARIO_WIDTH] float32 rows of NaN: every group keeps its random draw (bit-identical to no table)."""
    return torch.full((int(n), SCENARIO_WIDTH), float("nan"), dtype=torch.float32)


def fault_grid(n, rotors, onsets, effectiveness):
    """Rows whose fault group runs through the Cartesian product rotors x onsets x effectiveness (in that order, the last one
    fastest), tiled over the n envs: env i gets combination i % len(product).  Every other group is NaN.  Needs a task with
    rotorFault.enable; a rotor of -1 means no fault in that episode."""
    combos = list(itertools.product(rotors, onsets, effectiveness))
    if not combos:
        raise ValueError("fault_grid: rotors, onsets and effectiveness must not be empty")
    grid = torch.tensor(combos, dtype=torch.float32)
    rows = empty(n)
    rows[:, _ROTOR:_EFF + 1] = grid[torch.arange(int(n)) % len(combos)]
    return rows


def evaluate(env, act_fn, steps):
    """Run `steps` steps of `env` with actions `act_fn(obs_dict)` and count, per env, the episodes that finished, those that ended
    by time-out (survived) and the sum of their returns.  Accumulated on the device from reset_buf, timeout_buf and
    episode_return_buf; the loop never waits for the GPU.  Returns {"episodes", "survived"} (int64 [N]) and "return_sum"
    (float64 [N]), on the env's device."""
    n, dev = env.num_envs, env.device
    episodes = torch.zeros(n, dtype=torch.int64, device=dev)
    survived = torch.zeros(n, dtype=torch.int64, device=dev)
    return_sum = torch.zeros(n, dtype=torch.float64, device=dev)
    obs = env.obs_dict if env.obs_dict else {"obs": env.obs_buf}
    for _ in range(int(steps)):
        obs, _, _, _ = env.step(act_fn(obs))
        done = env.reset_buf != 0
        episodes += done
        survived += done & env.timeout_buf
        return_sum += torch.where(done, env.episode_return_buf.double(), 0.0)
    return {"episodes": episodes, "survived": survived, "return_sum": return_sum}
