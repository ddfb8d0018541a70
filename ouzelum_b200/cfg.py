"""Task configuration dictionaries mirroring the reference's Hydra YAML (isaacgymenvs/cfg/task/*.yaml).

hydra / omegaconf are not needed: `task_config(name, num_envs)` returns the plain nested dict the
reference's task constructors receive (`cfg["env"][...]`, `cfg["sim"][...]`), with the interpolations
(`${resolve_default:4096,${...num_envs}}`, `${eq:...}`) already resolved.  Keys under
`env` that the reference does not have (rotorFault, domainRandomization, linDrag, yawKm, seed, envIdBase,
collectMetrics, useCudaGraph) are this framework's zero-default extras (SURVEY.md 8a row P).
"""
import copy

_SIM = {"dt": 0.01, "substeps": 2, "up_axis": "z", "use_gpu_pipeline": True, "gravity": [0.0, 0.0, -9.81]}

_EXTRAS = {
    # mode "multi": rotors [lo, hi] faulted rotors per episode, the loss ramping in over rampSteps steps (include/ouzelum_b200.h)
    "rotorFault": {"enable": False, "mode": "single", "rotors": [1, 1], "effLow": 0.0, "effHigh": 0.5, "rampSteps": 0},
    "domainRandomization": {"enable": False, "low": 0.8, "high": 1.2},
    "linDrag": 0.0, "yawKm": 0.0,
    "POMDP": "none", "pomdp_prob": 0.0,
    "seed": 0, "envIdBase": 0, "collectMetrics": True, "useCudaGraph": False,
}

_TASKS = {
    # cfg/task/Ouzelum.yaml
    "Ouzelum": {"name": "Ouzelum", "physics_engine": "physx",
                "env": {"numEnvs": 4096, "envSpacing": 2.5, "maxEpisodeLength": 2000, "enableDebugVis": False,
                        "clipObservations": 5.0, "clipActions": 1.0, "enableCameraSensors": False},
                "sim": _SIM, "task": {"randomize": False}},
}
# cfg/task/{Lando,Landing,Landed,LeeLanded}.yaml differ from Ouzelum.yaml only in `name`
for _n in ("Lando", "Landing", "Landed", "LeeLanded"):
    _TASKS[_n] = copy.deepcopy(_TASKS["Ouzelum"])
    _TASKS[_n]["name"] = _n


# cfg/task/EKFLeeLanded.yaml
_TASKS["EKFLeeLanded"] = copy.deepcopy(_TASKS["Ouzelum"])
_TASKS["EKFLeeLanded"]["name"] = "EKFLeeLanded"
_TASKS["EKFLeeLanded"]["env"].update({"envSpacing": 5, "maxEpisodeLength": 700, "POMDP": "flicker", "pomdp_prob": 0.1,
                                      "ConvergenceTime": 300, "attach_pos_sensor": True, "attach_vel_sensor": True,
                                      "position_sensor_freq": 20, "velocity_sensor_freq": 75})
# cfg/task/Quadcopter.yaml
_TASKS["Quadcopter"] = {"name": "Quadcopter", "physics_engine": "physx",
                        "env": {"numEnvs": 8192, "envSpacing": 1.25, "maxEpisodeLength": 500, "enableDebugVis": False,
                                "clipObservations": 5.0, "clipActions": 1.0, "enableCameraSensors": False},
                        "sim": _SIM, "task": {"randomize": False}}


def task_names():
    return sorted(_TASKS)


def register_task_config(name, cfg):
    _TASKS[name] = cfg


def task_config(name, num_envs=None, **env_overrides):
    if name not in _TASKS:
        raise KeyError(f"unknown task {name!r}; known: {task_names()}")
    cfg = copy.deepcopy(_TASKS[name])
    for k, v in _EXTRAS.items():
        cfg["env"].setdefault(k, copy.deepcopy(v))
    if num_envs is not None:
        cfg["env"]["numEnvs"] = int(num_envs)          # isaacgymenvs/__init__.py:38
    for k, v in env_overrides.items():
        if isinstance(v, dict) and isinstance(cfg["env"].get(k), dict):
            cfg["env"][k].update(v)
        else:
            cfg["env"][k] = v
    return cfg
