"""`Env` / `VecTask`: the reference's vectorised-task surface on top of the fused CUDA step.

Mirrors isaacgymenvs/tasks/base/vec_task.py:60-406 -- same constructor signature, attributes
(`num_envs num_obs num_acts num_states observation_space action_space state_space device rl_device
obs_buf rew_buf reset_buf progress_buf timeout_buf randomize_buf states_buf extras control_freq_inv
max_episode_length`), same `step / reset / reset_done / reset_idx / get_state / zero_actions`
contracts -- so the reference's trainers (e.g. isaacgymenvs/RPO-LSTM/main.py:41-58,81,102) run
unchanged.  What differs: `step` is ONE kernel launch (no pre/post hooks, no host syncs, no
`gym.simulate`), and there is no CPU pipeline.
"""
from typing import Any, Dict, Tuple

import numpy as np
import torch

from .spaces import Box

import os as _os
_NVTX = _os.environ.get("OUZELUM_B200_NVTX", "0") == "1"


class Env:
    def __init__(self, config: Dict[str, Any], rl_device: str, sim_device: str, graphics_device_id: int, headless: bool):
        split_device = str(sim_device).split(":")
        self.device_type = split_device[0]
        self.device_id = int(split_device[1]) if len(split_device) > 1 else 0
        if self.device_type.lower() not in ("cuda", "gpu"):
            # vec_task.py:74-81 falls back to the CPU pipeline here; this framework has none.
            raise RuntimeError(f"sim_device={sim_device!r}: ouzelum_b200 has no CPU pipeline (sm_100a CUDA only)")
        self.device = "cuda:" + str(self.device_id)
        self.rl_device = rl_device
        self._tdev = torch.device(self.device)
        self._rl_on_sim_device = torch.device(rl_device) == self._tdev
        self.headless = headless
        self.graphics_device_id = -1 if headless else graphics_device_id

        self.num_environments = config["env"]["numEnvs"]
        self.num_agents = config["env"].get("numAgents", 1)
        self.num_observations = config["env"]["numObservations"]
        self.num_states = config["env"].get("numStates", 0)
        self.num_actions = config["env"]["numActions"]
        self.control_freq_inv = config["env"].get("controlFrequencyInv", 1)

        self.obs_space = Box(np.ones(self.num_obs) * -np.inf, np.ones(self.num_obs) * np.inf)
        self.state_space = Box(np.ones(self.num_states) * -np.inf, np.ones(self.num_states) * np.inf)
        self.act_space = Box(np.ones(self.num_actions) * -1., np.ones(self.num_actions) * 1.)

        self.clip_obs = config["env"].get("clipObservations", np.inf)
        self.clip_actions = config["env"].get("clipActions", np.inf)

    @property
    def observation_space(self):
        return self.obs_space

    @property
    def action_space(self):
        return self.act_space

    @property
    def num_envs(self) -> int:
        return self.num_environments

    @property
    def num_acts(self) -> int:
        return self.num_actions

    @property
    def num_obs(self) -> int:
        return self.num_observations


class VecTask(Env):
    metadata = {"render.modes": ["human", "rgb_array"], "video.frames_per_second": 24}
    reward_range = (-float("inf"), float("inf"))
    spec = None
    _states_from_kernel = False        # True once the task's step kernel writes states_buf (env.asymmetric_observations)

    def __init__(self, config, rl_device, sim_device, graphics_device_id, headless,
                 virtual_screen_capture: bool = False, force_render: bool = False):
        super().__init__(config, rl_device, sim_device, graphics_device_id, headless)
        self.cfg = config
        engine = config.get("physics_engine", "physx")
        if engine not in ("physx", "b200"):
            raise ValueError(f"Invalid physics engine backend: {engine}")          # vec_task.py:194-196
        up = config.get("sim", {}).get("up_axis", "z")
        if up != "z":
            raise ValueError(f"Invalid physics up-axis: {up}")                     # vec_task.py:454-457
        self.virtual_screen_capture = virtual_screen_capture
        self.force_render = force_render
        self.viewer = None
        self.dr_randomizations = {}
        self.first_randomization = True          # vec_task.py:137-141
        self.last_step = -1
        self.last_rand_step = -1
        self.sim_initialized = False
        self.create_sim()
        self.sim_initialized = True
        self.allocate_buffers()
        self.obs_dict = {}

    # ---- buffers (vec_task.py:254-277) --------------------------------------------------------------
    def allocate_buffers(self):
        dev = self.device
        self.obs_buf = torch.zeros((self.num_envs, self.num_obs), device=dev, dtype=torch.float)
        self.states_buf = torch.zeros((self.num_envs, self.num_states), device=dev, dtype=torch.float)
        self.rew_buf = torch.zeros(self.num_envs, device=dev, dtype=torch.float)
        self.reset_buf = torch.ones(self.num_envs, device=dev, dtype=torch.long)
        self.timeout_buf = torch.zeros(self.num_envs, device=dev, dtype=torch.bool)
        self.progress_buf = torch.zeros(self.num_envs, device=dev, dtype=torch.long)
        self.randomize_buf = torch.zeros(self.num_envs, device=dev, dtype=torch.long)
        self.extras = {}

    # ---- hooks a task implements --------------------------------------------------------------------
    def create_sim(self):
        raise NotImplementedError

    def _fused_step(self, actions: torch.Tensor):
        """Launch the task's fused step kernel: consumes `actions`, updates every *_buf in place."""
        raise NotImplementedError

    # ---- surface ------------------------------------------------------------------------------------
    def get_state(self):
        if self._states_from_kernel:       # clamped in the kernel: no torch op on the step path
            return self.states_buf if self._rl_on_sim_device else self.states_buf.to(self.rl_device)
        return torch.clamp(self.states_buf, -self.clip_obs, self.clip_obs).to(self.rl_device)

    def step(self, actions: torch.Tensor) -> Tuple[Dict[str, torch.Tensor], torch.Tensor, torch.Tensor, Dict[str, Any]]:
        """vec_task.py:313-359.  Action clamp, pre/post physics, reward, reset flags, time-outs and the
        observation clamp all happen inside the one kernel `_fused_step` launches."""
        if actions.dtype != torch.float32 or actions.device != self._tdev or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        if self.dr_randomizations:                  # vec_task.py:322-324: randomize actions (before the clamp, which is in the kernel)
            if "actions" in self.dr_randomizations:
                actions = self._noise_lambda("actions", actions.clone(), 0.0, 0)
        if _NVTX:                                   # OUZELUM_B200_NVTX=1: one NVTX range per env step (nsys / ncu --nvtx)
            torch.cuda.nvtx.range_push(f"{type(self).__name__}.step")
            self._fused_step(actions)
            torch.cuda.nvtx.range_pop()
        else:
            self._fused_step(actions)
        if self.dr_randomizations and "observations" in self.dr_randomizations:
            # vec_task.py:348-350: randomize observations, then the clamp of :353 (the kernel has already clamped the un-noised
            # observation: identical whenever that lies inside +-clip_obs)
            self._noise_lambda("observations", self.obs_buf, float(self.clip_obs), -1)
        if self._rl_on_sim_device:                  # the usual case: no `.to()` round trips through the dispatcher
            self.extras["time_outs"] = self.timeout_buf
            self.obs_dict["obs"] = self.obs_buf
            if self.num_states > 0:
                self.obs_dict["states"] = self.get_state()
            return self.obs_dict, self.rew_buf, self.reset_buf, self.extras
        self.extras["time_outs"] = self.timeout_buf.to(self.rl_device)
        self.obs_dict["obs"] = self.obs_buf.to(self.rl_device)
        if self.num_states > 0:
            self.obs_dict["states"] = self.get_state()
        return self.obs_dict, self.rew_buf.to(self.rl_device), self.reset_buf.to(self.rl_device), self.extras

    # ---- observation / action noise of the domain randomisation (vec_task.py:538-646) ----------------------------
    def _frame_count(self):
        """gym.get_frame_count(sim): control steps taken so far (the handle's device step counter when the task has one)."""
        sim = getattr(self, "sim", None)
        if sim is not None and hasattr(sim, "step_count"):
            return int(sim.step_count)
        if getattr(self, "_step_record", None) is not None:
            import ctypes as C
            from ._lib import check, lib
            out = C.c_uint64()
            check(lib.ozl_step_record_read(self._step_record.data_ptr(), C.byref(out), torch.cuda.current_stream().cuda_stream))
            return int(out.value)
        return 0

    def apply_randomizations(self, dr_params):
        """The non-physical part of `VecTask.apply_randomizations` (vec_task.py:538-646): builds the `observations` / `actions` noise
        lambdas -- gaussian or uniform, additive or scaling, linear / constant schedule, with the correlated component
        (`range_correlated`) that is re-drawn on every randomisation event and held in between.  `frequency` gates the events as in the
        reference (:546-566).  The physical parameters of `dr_params["actor_params"]` are randomised inside the step kernel at every
        reset (ozl_cfg.dr[], set from the task config at construction); `sim_params` (gravity) is not randomised here."""
        from ._lib import DR_ADDITIVE, DR_GAUSSIAN, DR_SCALING, DR_UNIFORM, OzlNoiseLambda
        rand_freq = dr_params.get("frequency", 1)
        self.last_step = self._frame_count()
        do_nonenv_randomize = True if self.first_randomization else (self.last_step - self.last_rand_step) >= rand_freq
        if do_nonenv_randomize:
            self.last_rand_step = self.last_step
        for name in ("observations", "actions"):
            if name in dr_params and do_nonenv_randomize:
                p = dr_params[name]
                dist, op = p["distribution"], p["operation"]
                if dist not in ("gaussian", "uniform") or op not in ("additive", "scaling"):
                    raise ValueError(f"randomization_params[{name!r}]: distribution {dist!r} / operation {op!r} not supported "
                                     "(gaussian | uniform, additive | scaling)")
                sched = p["schedule"] if "schedule" in p else None
                sched_step = p["schedule_steps"] if "schedule" in p else None
                if sched == "linear":
                    s = 1.0 / sched_step * min(self.last_step, sched_step)
                elif sched == "constant":
                    s = 0 if self.last_step < sched_step else 1
                else:
                    s = 1
                a, b = p["range"]
                ac, bc = p.get("range_correlated", [0.0, 0.0])
                if op == "additive":
                    a, b, ac, bc = a * s, b * s, ac * s, bc * s
                elif dist == "gaussian":
                    b, a = b * s, a * s + 1.0 * (1.0 - s)
                    bc, ac = bc * s, ac * s + 1.0 * (1.0 - s)
                else:
                    a, b = a * s + 1.0 * (1.0 - s), b * s + 1.0 * (1.0 - s)
                    ac, bc = ac * s + 1.0 * (1.0 - s), bc * s + 1.0 * (1.0 - s)
                spec = OzlNoiseLambda(DR_GAUSSIAN if dist == "gaussian" else DR_UNIFORM,
                                      DR_ADDITIVE if op == "additive" else DR_SCALING, a, b, ac, bc)
                keys = ("mu", "var", "mu_corr", "var_corr") if dist == "gaussian" else ("lo", "hi", "lo_corr", "hi_corr")
                self.dr_randomizations[name] = dict(zip(keys, (a, b, ac, bc)), spec=spec, corr_epoch=int(self.last_step),
                                                    distribution=dist, operation=op)
        self.first_randomization = False

    def _noise_lambda(self, name, tensor, clip, step_offset):
        """Apply the `name` lambda in place (one launch).  The step index comes from the task's device step counter when it has one
        (CUDA-graph capturable); `step_offset` = -1 for the observations, which are noised after the step has advanced it."""
        import ctypes as C
        from ._lib import check, lib
        d = self.dr_randomizations[name]
        ptr_, host_step = self._step_record_ptr(), 0
        if not ptr_:
            raise RuntimeError("noise lambdas need a task with a device step counter")
        seed = int(self.cfg["env"].get("seed", 0)) if isinstance(self.cfg, dict) else 0
        base = int(self.cfg["env"].get("envIdBase", 0)) if isinstance(self.cfg, dict) else 0
        check(lib.ozl_noise_lambda_apply(tensor.shape[0], tensor.shape[1], tensor.data_ptr(), C.byref(d["spec"]), clip, seed,
                                         host_step, ptr_, step_offset, d["corr_epoch"], base, 0 if name == "observations" else 1,
                                         torch.cuda.current_stream().cuda_stream))
        return tensor

    def _step_record_ptr(self):
        """Device address of the task's step-counter record (0 when the task keeps its step index on the host)."""
        if getattr(self, "_step_rec_ptr", None) is None:
            import ctypes as C
            from ._lib import check, lib
            sim = getattr(self, "sim", None)
            p = C.c_void_p()
            if sim is not None and hasattr(sim, "_h"):
                check(lib.ozl_step_counter_ptr(sim._h, C.byref(p)))
            elif getattr(self, "_step_record", None) is not None:      # Quadcopter: stand-alone record (ozl_step_record_init)
                p = C.c_void_p(self._step_record.data_ptr())
            self._step_rec_ptr = p.value or 0
        return self._step_rec_ptr

    def zero_actions(self) -> torch.Tensor:
        return torch.zeros([self.num_envs, self.num_actions], dtype=torch.float32, device=self.rl_device)

    def reset_idx(self, env_idx):
        pass

    def reset(self):
        """vec_task.py:377-389: returns the (initially zero) observation buffer; no simulation."""
        self.obs_dict["obs"] = torch.clamp(self.obs_buf, -self.clip_obs, self.clip_obs).to(self.rl_device)
        if self.num_states > 0:
            self.obs_dict["states"] = self.get_state()
        return self.obs_dict

    def reset_done(self):
        """vec_task.py:391-406."""
        done_env_ids = self.reset_buf.nonzero(as_tuple=False).flatten()
        if len(done_env_ids) > 0:
            self.reset_idx(done_env_ids)
        self.obs_dict["obs"] = torch.clamp(self.obs_buf, -self.clip_obs, self.clip_obs).to(self.rl_device)
        if self.num_states > 0:
            self.obs_dict["states"] = self.get_state()
        return self.obs_dict, done_env_ids

    def render(self, mode="rgb_array"):
        return None                      # headless only: no viewer in this framework

    def close(self):
        pass

    @property
    def unwrapped(self):
        return self
