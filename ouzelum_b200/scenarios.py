"""Scenario tables: per-env episode conditions that every reset applies in place of the random draws (`X500Task.set_scenarios`,
C ABI `ozl_set_scenarios`; row layout OZL_SCN_* in include/ouzelum_b200.h, `_lib.SCENARIO_LAYOUT`).

    rows = scenarios.fault_grid(env.num_envs, rotors=[0, 1, 2, 3], onsets=[0, 300], effectiveness=[0.1, 0.5])
    env.set_scenarios(rows)
    result = scenarios.evaluate(env, lambda obs: policy(obs["obs"]), steps=4000)

Two policies evaluated on the same table see the same faults, spawn poses and body parameters in every episode.
`run_episodes(env, act_fn, steps)` returns the episode-log record (termination cause and conditions) of every episode of a run.
"""
import itertools

import torch

from ._lib import SCENARIO_LAYOUT, SCENARIO_WIDTH

_ROTOR, _ONSET, _EFF = (SCENARIO_LAYOUT[k] for k in ("OZL_SCN_FAULT_ROTOR", "OZL_SCN_FAULT_ONSET", "OZL_SCN_FAULT_EFF"))
_RONSET, _REFF = SCENARIO_LAYOUT["OZL_SCN_RFAULT_ONSET"], SCENARIO_LAYOUT["OZL_SCN_RFAULT_EFF"]


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


def multi_fault_grid(n, effectiveness, onsets):
    """Rows whose rotor-faults group (rotorFault.mode "multi") runs through effectiveness x onsets (the last one fastest), tiled
    over the n envs like `fault_grid`: `effectiveness` is a list of 4-tuples (e_0..e_3, each in [0, 1]; (1, 1, 1, 1) means no
    fault in that episode).  Every other group is NaN."""
    combos = [tuple(float(x) for x in e) + (float(o),) for e, o in itertools.product(effectiveness, onsets)]
    if not combos:
        raise ValueError("multi_fault_grid: effectiveness and onsets must not be empty")
    if any(len(c) != 5 for c in combos):
        raise ValueError("multi_fault_grid: every effectiveness entry must have four values (rotors 0..3)")
    grid = torch.tensor([(c[4],) + c[:4] for c in combos], dtype=torch.float32)       # onset, e_0..e_3 (slot order)
    rows = empty(n)
    rows[:, _RONSET:_REFF + 4] = grid[torch.arange(int(n)) % len(combos)]
    return rows


def run_episodes(env, act_fn, steps, capacity=None):
    """Run `steps` steps of `env` with actions `act_fn(obs_dict)` and return the episode-log records (`X500Task.episode_log`) of
    every episode that ended during the run, concatenated in (step, env) order, with "dropped" 0.  An env ends at most one episode
    per step, so the log (of `capacity` records, default 64 per env) is drained every capacity // num_envs steps and loses none.
    A log the env had enabled is replaced by this run's and disabled at the end."""
    n = env.num_envs
    capacity = 64 * n if capacity is None else int(capacity)
    if capacity < n:
        raise ValueError(f"run_episodes: capacity {capacity} is below one record per env ({n})")
    every = capacity // n
    env.enable_episode_log(capacity)
    parts = []
    try:
        obs = env.obs_dict if env.obs_dict else {"obs": env.obs_buf}
        for t in range(int(steps)):
            obs, _, _, _ = env.step(act_fn(obs))
            if (t + 1) % every == 0:
                parts.append(env.episode_log(clear=True))
        parts.append(env.episode_log(clear=True))
    finally:
        env.disable_episode_log()
    out = {k: torch.cat([p[k] for p in parts]) for k in parts[0] if k != "dropped"}
    out["dropped"] = sum(p["dropped"] for p in parts)
    return out


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
