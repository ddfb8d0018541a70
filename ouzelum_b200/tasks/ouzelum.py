"""`Ouzelum`: x500 quadcopter tracking a randomly re-sampled waypoint, as ONE fused kernel per step.

Mirror of isaacgymenvs/tasks/ouzelum.py (class surface :40-99, hooks :180-295, reward :302-332).
The reference builds an Isaac Gym sim with an O(N) Python loop (:153-168) and steps it with ~45
eager launches + 3 host syncs + PhysX; here `create_sim` allocates the SoA state through the C ABI
and `step` is a single `ozl_step` launch with no host synchronisation.
"""
import math

import torch

from .. import _lib
from ..sim import QuadSim
from ..vec_task import VecTask

_POMDP = {"none": 0, None: 0, "flicker": 1, "random_noise": 2, "flickering_and_random_noise": 3}
_DR_DIST = {"uniform": _lib.DR_UNIFORM, "loguniform": _lib.DR_LOGUNIFORM, "gaussian": _lib.DR_GAUSSIAN}
_DR_OP = {"scaling": _lib.DR_SCALING, "additive": _lib.DR_ADDITIVE}
_DR_SCHED = {None: _lib.DR_SCHED_NONE, "linear": _lib.DR_SCHED_LINEAR, "constant": _lib.DR_SCHED_CONSTANT}
# reference attribute names (gymapi.RigidBodyProperties: mass, inertia) and this framework's rotor parameters
_DR_NAMES = {"mass": "mass", "ixx": "ixx", "iyy": "iyy", "izz": "izz", "arm": "arm", "thrust_scale": "thrust_scale",
             "yaw_km": "yaw_km", "motor_constant": "yaw_km"}


def dr_spec(attr_params):
    """One attribute block of the reference's `randomization_params` (isaacgymenvs/utils/dr_utils.py:71-81:
    range / distribution / operation / schedule / schedule_steps) -> ozl_dr_param tuple."""
    dist, op = attr_params["distribution"], attr_params["operation"]
    if dist not in _DR_DIST:
        raise ValueError(f"unknown randomization distribution {dist!r} (uniform, loguniform, gaussian)")
    if op not in _DR_OP:
        raise ValueError(f"unknown randomization operation {op!r} (scaling, additive)")
    sched = attr_params.get("schedule")
    if sched not in _DR_SCHED:
        raise ValueError(f"unknown randomization schedule {sched!r} (linear, constant)")
    lo, hi = attr_params["range"]
    return (_DR_DIST[dist], _DR_OP[op], float(lo), float(hi), _DR_SCHED[sched], int(attr_params.get("schedule_steps", 0) or 0))


def dr_from_task_cfg(cfg):
    """Domain-randomisation schema of a task dict -> (enable, {parameter: spec}).  Two spellings are accepted:
      * the reference's: cfg["task"]["randomize"] = True and cfg["task"]["randomization_params"]["actor_params"][<actor>]
        ["rigid_body_properties" | "rotor_properties"][<attr>] = {range, operation, distribution[, schedule, schedule_steps]}
        (cfg/task/*.yaml of the stock tasks; applied at resets, tasks/base/vec_task.py:538-768) with attrs
        mass / ixx / iyy / izz / arm / thrust_scale / yaw_km (alias motor_constant);
      * the shorthand env["domainRandomization"] = {enable, low, high}: scaling x uniform [low, high) on mass, inertia, arm, thrust scale."""
    env, task = cfg["env"], cfg.get("task", {}) or {}
    out = {}
    short = env.get("domainRandomization", {}) or {}
    enable = bool(short.get("enable", False))
    if enable:
        lo, hi = float(short.get("low", 0.8)), float(short.get("high", 1.2))
        for name in ("mass", "ixx", "iyy", "izz", "arm", "thrust_scale"):
            out[name] = (_lib.DR_UNIFORM, _lib.DR_SCALING, lo, hi, 0, 0)
    if task.get("randomize", False):
        actors = (task.get("randomization_params", {}) or {}).get("actor_params", {}) or {}
        if actors and not enable:
            # the reference randomises only what the YAML lists
            for name in ("mass", "ixx", "iyy", "izz", "arm", "thrust_scale", "yaw_km"):
                out[name] = (_lib.DR_NONE, _lib.DR_SCALING, 1.0, 1.0, 0, 0)
        for actor, props in actors.items():
            for group in ("rigid_body_properties", "rotor_properties"):
                for attr, ap in (props.get(group, {}) or {}).items():
                    if attr not in _DR_NAMES:
                        raise ValueError(f"randomization_params: attribute {attr!r} of actor {actor!r} is not randomisable here "
                                         f"(known: {sorted(_DR_NAMES)})")
                    out[_DR_NAMES[attr]] = dr_spec(ap)
                    enable = True
    return enable, out


def rotor_fault_cfg(fault):
    """env["rotorFault"] = {enable, mode: "single" | "multi", rotors: [lo, hi], effLow, effHigh, rampSteps} -> ozl_cfg fields.
    "single" (the default) is fault_mode 1; "multi" is fault_mode 2 (several rotors, gradual loss: include/ouzelum_b200.h)."""
    fault = fault or {}
    mode = fault.get("mode", "single")
    if mode not in ("single", "multi"):
        raise ValueError(f"rotorFault.mode must be 'single' or 'multi', got {mode!r}")
    lo_e, hi_e = float(fault.get("effLow", 0.0)), float(fault.get("effHigh", 0.5))
    kw = dict(fault_mode=(2 if mode == "multi" else 1) if fault.get("enable", False) else 0, fault_eff_lo=lo_e, fault_eff_range=hi_e - lo_e)
    rotors, ramp = fault.get("rotors", [1, 1]), fault.get("rampSteps", 0)
    if mode == "multi":
        if len(rotors) != 2 or any(int(r) != r for r in rotors) or not 0 <= rotors[0] <= rotors[1] <= 4:
            raise ValueError(f"rotorFault.rotors must be [lo, hi] with integers 0 <= lo <= hi <= 4, got {rotors!r}")
        if int(ramp) != ramp or not 0 <= ramp < 1 << 24:
            raise ValueError(f"rotorFault.rampSteps must be an integer in [0, 2^24), got {ramp!r}")
        if not 0.0 <= lo_e <= hi_e <= 1.0:
            raise ValueError(f"rotorFault: multi needs 0 <= effLow <= effHigh <= 1, got {lo_e}, {hi_e}")
    kw.update(fault_rotors_lo=int(rotors[0]), fault_rotors_hi=int(rotors[1]), fault_ramp_steps=int(ramp))
    return kw


def refuse_multi_fault(task_name, env_cfg):
    """rotorFault.mode "multi" (fault_mode 2) is applied by the rotor-actuated step kernels only: a task whose step is
    wrench-actuated or has a kernel of its own raises ValueError for it."""
    if (env_cfg.get("rotorFault", {}) or {}).get("mode", "single") == "multi":
        raise ValueError(f"{task_name}: rotorFault.mode 'multi' is not supported (its step does not apply per-rotor faults)")


def decode_episode_records(rows):
    """[k, EPLOG_WIDTH] float32 records (layout OZL_EPLOG_* in include/ouzelum_b200.h) -> dict of named tensors, sorted by (step,
    env).  The row contents are deterministic; their order in the buffer is not."""
    L = _lib.EPLOG_LAYOUT
    bits = rows.view(torch.int32)
    env = bits[:, L["OZL_EPLOG_ENV"]].long() & 0xFFFFFFFF
    s = L["OZL_EPLOG_STEP"]
    step = (bits[:, s + 1].long() << 32) | (bits[:, s].long() & 0xFFFFFFFF)
    order = torch.argsort(env, stable=True)                    # two stable passes: env, then step (a packed key would overflow)
    order = order[torch.argsort(step[order], stable=True)]
    rows, bits, env, step = rows[order], bits[order], env[order], step[order]
    flags = bits[:, L["OZL_EPLOG_FLAGS"]]
    col = lambda name, k=1: rows[:, L[name]:L[name] + k].clone()
    return {"env": env, "length": bits[:, L["OZL_EPLOG_LENGTH"]].long(), "step": step,
            "return": rows[:, L["OZL_EPLOG_RETURN"]].clone(),
            "timeout": (flags & 1) != 0, "crash_dist": (flags & 2) != 0, "crash_z": (flags & 4) != 0, "landed": (flags & 8) != 0,
            "fault_active": (flags & 16) != 0, "onset": bits[:, L["OZL_EPLOG_ONSET"]].long(), "dist": rows[:, L["OZL_EPLOG_DIST"]].clone(),
            "eff": col("OZL_EPLOG_EFF", 4), "params": col("OZL_EPLOG_MASS", 7), "pos": col("OZL_EPLOG_POS", 3),
            "linvel": col("OZL_EPLOG_LINVEL", 3), "target": col("OZL_EPLOG_TARGET", 3)}


def x500_cfg_from_task(cfg, num_envs, **over):
    """Translate the reference-style nested task dict into the C `ozl_cfg`."""
    env, sim = cfg["env"], cfg.get("sim", {})
    dt = float(sim.get("dt", 0.01))
    fault = env.get("rotorFault", {}) or {}
    dr_enable, dr = dr_from_task_cfg(cfg)
    pomdp = env.get("POMDP", "none")
    if pomdp not in _POMDP:
        # isaacgymenvs/utils/POMDP.py:19-20
        raise ValueError("pomdp was not in ['flicker', 'random_noise', 'flickering_and_random_noise']!")
    kw = dict(
        env_id_base=int(env.get("envIdBase", 0)), seed=int(env.get("seed", 0)),
        max_episode_length=int(env["maxEpisodeLength"]),
        substeps=int(sim.get("substeps", 2)), control_freq_inv=int(env.get("controlFrequencyInv", 1)),
        dt=dt, gravity_z=float(sim.get("gravity", [0, 0, -9.81])[2]),
        clip_actions=float(min(env.get("clipActions", math.inf), 3.0e38)),
        clip_obs=float(min(env.get("clipObservations", math.inf), 3.0e38)),
        thrust_rate=dt * 2000,                         # ouzelum.py:237-238
        lin_drag=float(env.get("linDrag", 0.0)), yaw_km=float(env.get("yawKm", 0.0)),
        **rotor_fault_cfg(fault),
        dr_enable=1 if dr_enable else 0, dr=dr,
        pomdp_mode=_POMDP[pomdp], pomdp_prob=float(env.get("pomdp_prob", 0.0)),
        noise_sigma=float(env.get("pomdp_prob", 0.0)),  # POMDP.py:8-9: one knob feeds both
        collect_metrics=1 if env.get("collectMetrics", True) else 0,
    )
    kw.update(over)
    return _lib.default_cfg(num_envs, **kw)


def asymmetric_states(task_name, env_cfg, supported):
    """`env.asymmetric_observations` (the stock IsaacGymEnvs name of the numStates critic input): True -> set numStates to the
    kernel's privileged-state width before VecTask reads it.  Raises ValueError for a task whose step kernel has no states output
    or for an explicit numStates of another width."""
    if not bool(env_cfg.get("asymmetric_observations", False)):
        return False
    if not supported:
        raise ValueError(f"{task_name}: asymmetric_observations is not supported (its step kernel does not write a states output)")
    ns = env_cfg.get("numStates")
    if ns is not None and int(ns) != _lib.STATES_WIDTH:
        raise ValueError(f"{task_name}: asymmetric_observations writes {_lib.STATES_WIDTH} states per env, but numStates = {ns}")
    env_cfg["numStates"] = _lib.STATES_WIDTH
    return True


class X500Task(VecTask):
    """Shared machinery of the x500 tasks: owns the `QuadSim` handle and launches the fused step."""

    num_x500_obs = 13
    num_x500_actions = 4
    supports_states = True             # the step kernels can write the privileged critic state (ozl_set_states_output)
    supports_scenarios = True          # the step kernels can apply a scenario table at resets (ozl_set_scenarios)
    supports_episode_log = True        # the step kernels can append a record per finished episode (ozl_set_episode_log)

    def __init__(self, cfg, rl_device, sim_device, graphics_device_id, headless,
                 virtual_screen_capture=False, force_render=False):
        self.cfg = cfg
        self.max_episode_length = self.cfg["env"]["maxEpisodeLength"]
        self.debug_viz = self.cfg["env"].get("enableDebugVis", False)
        self.cfg["env"]["numObservations"] = self.num_x500_obs     # ouzelum.py:50
        self.cfg["env"]["numActions"] = self.num_x500_actions      # ouzelum.py:55
        asym = asymmetric_states(type(self).__name__, self.cfg["env"], self.supports_states)
        super().__init__(config=self.cfg, rl_device=rl_device, sim_device=sim_device,
                         graphics_device_id=graphics_device_id, headless=headless,
                         virtual_screen_capture=virtual_screen_capture, force_render=force_render)
        if asym:                       # registered once: the buffer never moves, so captured graphs keep writing it
            self.sim.set_states_output(self.states_buf)
            self._states_from_kernel = True
        self.dt = float(self.cfg.get("sim", {}).get("dt", 0.01))
        self._timeout_u8 = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
        self.timeout_buf = self._timeout_u8.view(torch.bool)
        # RecordEpisodeStatisticsTorch "r"/"l" equivalents (RPO-LSTM/utils.py:24-30), filled by the kernel
        self.episode_return_buf = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
        self._host_io, self._host_keep = {}, []          # step_host: argument blocks cached by actions-buffer address
        self._graph = None
        self._static_actions = None
        self.scenarios = None          # the registered scenario table (CPU copy), see set_scenarios
        self._eplog = None             # (records, head) of the episode log, see enable_episode_log
        self.use_cuda_graph = bool(self.cfg["env"].get("useCudaGraph", False))

    # ---- overridable pieces --------------------------------------------------------------------------
    def _native_cfg(self):
        return x500_cfg_from_task(self.cfg, self.num_envs)

    def create_sim(self):
        self.native_cfg = self._native_cfg()
        self.sim = QuadSim(self.native_cfg, self.device)

    # ---- fused step ------------------------------------------------------------------------------------
    def _launch(self, actions):
        self.sim.step(actions, self.obs_buf, self.rew_buf, self.reset_buf, self.progress_buf,
                      self._timeout_u8, self.episode_return_buf)

    def _fused_step(self, actions):
        if not self.use_cuda_graph:
            self._launch(actions)
            return
        if self._graph is None:
            self._static_actions = torch.empty_like(actions)
            self._static_actions.copy_(actions)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._launch(self._static_actions)
            self._graph = g
        self._static_actions.copy_(actions)
        self._graph.replay()

    # ---- host-consumer step ----------------------------------------------------------------------------------
    def step_host(self, actions_host):
        """`step` for a consumer that lives on the CPU (rl_device == "cpu" in the reference's terms, vec_task.py:353-359):
        `actions_host` is a pinned [N,4] float32 CPU tensor; returns pinned CPU tensors (obs [N,13] f32, reward [N] f32,
        reset [N] int64 -- the reference's dtypes) that are valid when the call returns.  The kernel reads / writes them in place
        across PCIe (zero-copy).  `host_done_u8` holds the same flags as one byte per env."""
        io = self._host_io.get(actions_host.data_ptr())
        if io is None:
            io = self._make_host_io(actions_host)
        # one foreign call: launch + stream synchronise (ozl_step_host_sync)
        if _lib.lib.ozl_step_host_sync(self.sim._h, io, torch._C._cuda_getCurrentRawStream(self.sim.index)):
            _lib.check(1)
        return self._h_obs, self._h_rew, self._h_reset

    def step_host_async(self, actions_host, stream=None):
        """Launch-only half of `step_host` (EnvPool-style pipelining: a CPU consumer that splits its envs over two task objects can
        let one object's PCIe write-back overlap the other's action reads and compute).  The results are valid after
        `step_host_wait()`.  `stream`: a torch.cuda.Stream to launch on (default: the current stream)."""
        io = self._host_io.get(actions_host.data_ptr())
        if io is None:
            io = self._make_host_io(actions_host)
        self._host_stream = stream.cuda_stream if stream is not None else torch._C._cuda_getCurrentRawStream(self.sim.index)
        if _lib.lib.ozl_step_host_launch(self.sim._h, io, self._host_stream):
            _lib.check(1)

    def step_host_wait(self):
        if _lib.lib.ozl_step_host_wait(self.sim._h, self._host_stream):
            _lib.check(1)
        return self._h_obs, self._h_rew, self._h_reset

    @property
    def host_done_u8(self):
        """The reset flags of the last host step, one byte per env (pinned CPU tensor)."""
        return self._h_done

    def _make_host_io(self, actions_host):
        """Argument block of ozl_step_host_sync for one actions buffer, validated once and cached by address."""
        import ctypes as C
        from .._lib import OzlHostIo
        if not hasattr(self, "_h_obs"):
            pin = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt).pin_memory()
            self._h_obs, self._h_rew = pin(self.num_envs, self.num_obs), pin(self.num_envs)
            self._h_done = pin(self.num_envs, dt=torch.uint8)
            self._h_reset = pin(self.num_envs, dt=torch.int64)          # reset_buf in the reference's dtype (vec_task.py:353-359)
        if len(self._host_keep) >= 64:                       # a caller that passes a fresh buffer every step
            self._host_io.clear()
            self._host_keep.clear()
        if not actions_host.is_pinned() or actions_host.dtype != torch.float32 or not actions_host.is_contiguous() \
                or tuple(actions_host.shape) != (self.num_envs, self.num_acts):
            raise ValueError("step_host needs a contiguous page-locked (pinned) float32 CPU tensor of shape [num_envs, num_acts]")
        io = OzlHostIo(actions_host.data_ptr(), self._h_obs.data_ptr(), self._h_rew.data_ptr(), self._h_done.data_ptr(),
                       self._h_reset.data_ptr(), self.reset_buf.data_ptr(), self.progress_buf.data_ptr(), self._timeout_u8.data_ptr(),
                       self.episode_return_buf.data_ptr())
        ref = C.byref(io)
        self._host_keep.append((io, actions_host))          # keep the struct and the caller's buffer alive
        self._host_io[actions_host.data_ptr()] = ref
        return ref

    # ---- reference-style state views (copies out of the private SoA state) ------------------------------
    @property
    def root_states(self):
        return self.sim.get_state()["root"]

    @property
    def root_positions(self):
        return self.root_states[:, 0:3]

    @property
    def root_quats(self):
        return self.root_states[:, 3:7]

    @property
    def root_linvels(self):
        return self.root_states[:, 7:10]

    @property
    def root_angvels(self):
        return self.root_states[:, 10:13]

    @property
    def thrusts(self):
        return self.sim.get_state()["thrust"]

    @property
    def target_root_positions(self):
        return self.sim.get_state()["target"]

    def set_root_states(self, root):
        self.sim.set_state(root=root)

    # ---- scenario table ----------------------------------------------------------------------------------------------------
    def set_scenarios(self, rows):
        """Pin per-env episode conditions: from now on every reset of env i applies row i of `rows` (float32 [num_envs,
        SCENARIO_WIDTH] on CPU or CUDA, layout `_lib.SCENARIO_LAYOUT` / OZL_SCN_* in include/ouzelum_b200.h) in place of the random
        draws -- spawn pose, velocities, target, rotor-fault schedule, body parameters.  An all-NaN group keeps the draw
        (`ouzelum_b200.scenarios.empty`).  Not pinned: the per-step sensor-fault draws, the observation / action noise and the
        ground vehicle's trajectory.  New contents reach a captured CUDA graph at its next resets; registering or unregistering
        (rows = None) re-captures this task's own step graph.  Raises ValueError for an invalid table."""
        if not self.supports_scenarios:
            raise ValueError(f"{type(self).__name__}: scenario tables are not supported (its step kernel does not apply them)")
        host = None
        if rows is not None:
            if not isinstance(rows, torch.Tensor):
                raise ValueError("scenario rows must be a torch.Tensor")
            host = rows.detach().to("cpu").contiguous()
            self._check_scenarios(host)
        self.sim.set_scenarios(host)
        if (host is None) != (self.scenarios is None):
            self._graph = None         # the captured step holds the kernels without (or with) the table
        self.scenarios = None if host is None else host.clone()

    def _check_scenarios(self, rows):
        """Task-specific refusals of a scenario table (the library validates the rows themselves)."""

    # ---- episode log -------------------------------------------------------------------------------------------------------
    def enable_episode_log(self, capacity):
        """From now on every step appends one record per episode that ends -- termination cause, length, return, and the episode's
        conditions (fault onset and per-rotor effectiveness, body parameters, final position, velocity and target) -- to a device
        buffer of `capacity` records; `episode_log()` reads and clears it.  Records beyond the capacity are counted and dropped.
        Re-captures this task's own step graph.  The log is not env state: checkpoints do not carry it."""
        if not self.supports_episode_log:
            raise ValueError(f"{type(self).__name__}: the episode log is not supported (its step kernel writes no records)")
        capacity = int(capacity)
        if capacity < 1:
            raise ValueError(f"episode log capacity must be >= 1, got {capacity}")
        records = torch.zeros(capacity, _lib.EPLOG_WIDTH, dtype=torch.float32, device=self.device)
        head = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.sim.set_episode_log(records, head)
        self._eplog = (records, head)
        self._graph = None             # the captured step holds the kernels without (or with another) log

    def disable_episode_log(self):
        if self._eplog is None:
            return
        self.sim.set_episode_log(None, None)
        self._eplog = None
        self._graph = None

    def episode_log(self, clear=True):
        """The records since the last clearing read, as a dict of tensors on the env's device sorted by (step, env): "env",
        "length", "step" (int64 [k]), "return", "dist" (float32 [k]), the causes "timeout", "crash_dist", "crash_z", "landed" and
        "fault_active" (bool [k]), "onset" (int64 [k], -1: no fault scheduled), "eff" [k, 4], "params" [k, 7] (mass, ixx, iyy, izz,
        arm, thrust scale, yaw_km), "pos", "linvel", "target" [k, 3]; and "dropped", the number of records the capacity lost.  One
        host synchronisation; `clear` zeroes the count (stream-ordered)."""
        if self._eplog is None:
            raise ValueError("the episode log is not enabled (enable_episode_log)")
        records, head = self._eplog
        total = int(head.item())
        k = min(total, records.shape[0])
        out = decode_episode_records(records[:k])
        if clear:
            head.zero_()
        out["dropped"] = total - k
        return out

    def reset_idx(self, env_ids):
        """ouzelum.py:192-216.  The re-initialisation itself happens inside the next step's kernel (exactly when
        the reference's takes effect: pre_physics_step, ouzelum.py:226-229); here the request is recorded."""
        self.reset_buf[env_ids] = 1

    # ---- checkpoint / resume of the ENV state (the reference never saves it; SURVEY section 5) ----------------------------
    def state_dict(self):
        """Everything needed to continue bit-identically: private state, per-env parameters, RNG time axis, surface buffers."""
        st = self.sim.get_state()
        params, fault = self.sim.get_params()
        rotor_eff = self.sim.get_rotor_eff() if self.native_cfg.fault_mode == 2 else None
        torch.cuda.current_stream().synchronize()
        return {"root": st["root"].cpu(), "thrust": st["thrust"].cpu(), "target": st["target"].cpu(), "ep_ret": st["ep_ret"].cpu(),
                "params": params.cpu(), "fault": fault.cpu(), "step_count": self.sim.step_count,
                "reset_buf": self.reset_buf.cpu(), "progress_buf": self.progress_buf.cpu(), "obs_buf": self.obs_buf.cpu(),
                "rew_buf": self.rew_buf.cpu(), "timeout_buf": self._timeout_u8.cpu(), "episode_return_buf": self.episode_return_buf.cpu(),
                "seed": int(self.native_cfg.seed), "num_envs": self.num_envs, "task": type(self).__name__,
                **({"rotor_eff": rotor_eff.cpu()} if rotor_eff is not None else {}),
                "scenarios": None if self.scenarios is None else self.scenarios.clone(),
                **({"states_buf": self.states_buf.cpu()} if self.num_states > 0 else {})}

    def load_state_dict(self, sd):
        if sd["num_envs"] != self.num_envs:
            raise ValueError(f"checkpoint has {sd['num_envs']} envs, this env has {self.num_envs}")
        if sd["seed"] != int(self.native_cfg.seed):
            raise ValueError("checkpoint was taken with a different RNG seed")
        if (self.native_cfg.fault_mode == 2) != ("rotor_eff" in sd):     # refused before anything is loaded
            raise ValueError("checkpoint and env disagree on rotorFault.mode 'multi' (the per-rotor effectiveness)")
        self.sim.set_state(root=sd["root"], thrust=sd["thrust"], target=sd["target"], ep_ret=sd["ep_ret"])
        self.sim.set_params(sd["params"], sd["fault"])
        if "rotor_eff" in sd:
            self.sim.set_rotor_eff(sd["rotor_eff"])
        self.sim.step_count = sd["step_count"]
        self.reset_buf.copy_(sd["reset_buf"])
        self.progress_buf.copy_(sd["progress_buf"])
        self.obs_buf.copy_(sd["obs_buf"])
        self.rew_buf.copy_(sd["rew_buf"])
        if "timeout_buf" in sd:
            self._timeout_u8.copy_(sd["timeout_buf"])
            self.episode_return_buf.copy_(sd["episode_return_buf"])
        if self.num_states > 0 and "states_buf" in sd:
            self.states_buf.copy_(sd["states_buf"])
        if "scenarios" in sd and (sd["scenarios"] is not None or self.scenarios is not None):
            self.set_scenarios(sd["scenarios"])
        if sd.get("task", type(self).__name__) != type(self).__name__:
            raise ValueError(f"checkpoint of task {sd['task']!r} loaded into {type(self).__name__!r}")
        self._graph = None

    def metrics(self, clear=False):
        """Episode / reward metrics vector accumulated in-kernel (see include/ouzelum_b200.h)."""
        return self.sim.metrics(clear=clear)

    def close(self):
        self.sim.close()


class Ouzelum(X500Task):
    """isaacgymenvs/tasks/ouzelum.py: target re-sampled in a 10x10x1 box every 500 steps, die z<0.5 or dist>8."""
