"""`QuadSim`: thin Python owner of one `ozl_env` handle (the private SoA state of N envs on one GPU).

It replaces what the reference obtains from Isaac Gym (`gymapi.acquire_gym()`, `create_sim`,
`acquire_actor_root_state_tensor` ... isaacgymenvs/tasks/ouzelum.py:59-99,112-178 and
isaacgymenvs/tasks/base/vec_task.py:189-221).  All tensors that cross the boundary are owned by the
caller (torch); PyTorch here is device memory + streams, not the compute path.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import check, lib, ptr


def _stream():
    # raw handle of torch's current stream on the current device (the fast path of torch.cuda.current_stream().cuda_stream)
    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())


class QuadSim:
    def __init__(self, cfg: _lib.OzlCfg, device="cuda:0"):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("ouzelum_b200 runs on CUDA (sm_100a) only: there is no CPU pipeline "
                               f"(got device {device!r}).")
        if not torch.cuda.is_available():
            raise RuntimeError("ouzelum_b200: no CUDA device is visible and there is no CPU fallback.")
        self.device = dev
        self.index = dev.index if dev.index is not None else torch.cuda.current_device()
        self.cfg = cfg
        self.num_envs = int(cfg.num_envs)
        self._h = C.c_void_p()
        with torch.cuda.device(self.index):
            check(lib.ozl_create(C.byref(cfg), self.index, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib.ozl_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- hot path ---------------------------------------------------------------------------------------
    def step(self, actions, obs, rew, reset, progress, timeout=None, ep_ret=None):
        """One fused env step (ozl_step).  All arguments are contiguous CUDA tensors owned by the caller."""
        check(lib.ozl_step(self._h, actions.data_ptr(), obs.data_ptr(), rew.data_ptr(), reset.data_ptr(),
                           progress.data_ptr(), ptr(timeout), ptr(ep_ret), _stream()))

    def step_host(self, actions_host, obs_host, rew_host, done_host, reset, progress, timeout=None, ep_ret=None):
        """ozl_step_host: actions / obs / rew / done are PINNED host tensors accessed zero-copy by the kernel."""
        for t in (actions_host, obs_host, rew_host, done_host):
            if not t.is_pinned():
                raise ValueError("step_host needs page-locked (pinned) host tensors")
        check(lib.ozl_step_host(self._h, actions_host.data_ptr(), obs_host.data_ptr(), rew_host.data_ptr(),
                                done_host.data_ptr(), reset.data_ptr(), progress.data_ptr(), ptr(timeout), ptr(ep_ret), _stream()))

    def step_tracking(self, actions, target, obs, rew, reset, progress, timeout=None, ep_ret=None):
        """ozl_step_tracking: the target [N,3] is supplied by the caller (landing family)."""
        check(lib.ozl_step_tracking(self._h, actions.data_ptr(), target.data_ptr(), obs.data_ptr(), rew.data_ptr(),
                                    reset.data_ptr(), progress.data_ptr(), ptr(timeout), ptr(ep_ret), _stream()))

    def step_wrench(self, wrench, target, obs, rew, reset, progress, timeout=None, ep_ret=None):
        """ozl_step_wrench: actuation by a body wrench [N,4] = (fz, tx, ty, tz); target may be None."""
        check(lib.ozl_step_wrench(self._h, wrench.data_ptr(), ptr(target), obs.data_ptr(), rew.data_ptr(),
                                  reset.data_ptr(), progress.data_ptr(), ptr(timeout), ptr(ep_ret), _stream()))

    def set_states_output(self, states):
        """ozl_set_states_output: every later step launch also writes the privileged critic state into `states`
        ([N, STATES_WIDTH] f32 CUDA tensor, kept alive by the caller); None unregisters."""
        if states is not None and (tuple(states.shape) != (self.num_envs, _lib.STATES_WIDTH) or states.dtype != torch.float32
                                   or not states.is_contiguous() or states.device != self.device):
            raise ValueError(f"states must be a contiguous float32 [{self.num_envs}, {_lib.STATES_WIDTH}] tensor on {self.device}")
        check(lib.ozl_set_states_output(self._h, ptr(states), _lib.STATES_WIDTH))

    def set_scenarios(self, rows):
        """ozl_set_scenarios: from now on every reset of env i applies row i of `rows` ([N, SCENARIO_WIDTH] float32, CPU or CUDA;
        NaN groups keep the random draws) in place of the draws.  The rows are validated and copied; None unregisters."""
        if rows is None:
            check(lib.ozl_set_scenarios(self._h, None, _lib.SCENARIO_WIDTH, _stream()), ValueError)
            return
        if not isinstance(rows, torch.Tensor) or rows.dtype != torch.float32 or tuple(rows.shape) != (self.num_envs, _lib.SCENARIO_WIDTH):
            raise ValueError(f"scenario rows must be a float32 [{self.num_envs}, {_lib.SCENARIO_WIDTH}] tensor")
        host = rows.detach().to("cpu").contiguous()
        check(lib.ozl_set_scenarios(self._h, host.data_ptr(), _lib.SCENARIO_WIDTH, _stream()), ValueError)

    def set_episode_log(self, records, head):
        """ozl_set_episode_log: every later step launch appends the record of each episode it ends to `records` ([capacity,
        EPLOG_WIDTH] f32 CUDA tensor) and counts it in `head` (one int64 CUDA tensor, zeroed by the caller); both kept alive by the
        caller.  records = None unregisters."""
        if records is None:
            check(lib.ozl_set_episode_log(self._h, None, 0, None, _lib.EPLOG_WIDTH), ValueError)
            return
        if records.dim() != 2 or records.shape[1] != _lib.EPLOG_WIDTH or records.dtype != torch.float32 \
                or not records.is_contiguous() or records.device != self.device:
            raise ValueError(f"records must be a contiguous float32 [capacity, {_lib.EPLOG_WIDTH}] tensor on {self.device}")
        if head.numel() != 1 or head.dtype != torch.int64 or head.device != self.device:
            raise ValueError(f"head must be one int64 element on {self.device}")
        check(lib.ozl_set_episode_log(self._h, records.data_ptr(), records.shape[0], head.data_ptr(), _lib.EPLOG_WIDTH), ValueError)

    def rollout(self, k, obs, rew, reset, progress):
        check(lib.ozl_rollout(self._h, int(k), obs.data_ptr(), rew.data_ptr(), reset.data_ptr(), progress.data_ptr(),
                              _stream()))

    def apply_resets(self, reset):
        """ozl_apply_resets: make the pending resets visible in the private state without stepping (idempotent)."""
        check(lib.ozl_apply_resets(self._h, reset.data_ptr(), _stream()))

    def get_root(self, out):
        check(lib.ozl_get_state(self._h, out.data_ptr(), None, None, None, _stream()))
        return out

    def reset_all(self, seed=0):
        check(lib.ozl_reset_all(self._h, int(seed), _stream()))

    # ---- state access -----------------------------------------------------------------------------------
    def _new(self, *shape, dtype=torch.float32):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    def get_state(self):
        n = self.num_envs
        root, thrust, target, ep = self._new(n, 13), self._new(n, 4), self._new(n, 3), self._new(n)
        check(lib.ozl_get_state(self._h, root.data_ptr(), thrust.data_ptr(), target.data_ptr(), ep.data_ptr(), _stream()))
        return dict(root=root, thrust=thrust, target=target, ep_ret=ep)

    def set_state(self, root=None, thrust=None, target=None, ep_ret=None):
        def prep(t, *shape):
            if t is None:
                return None
            t = t.to(device=self.device, dtype=torch.float32).contiguous()
            if tuple(t.shape) != shape:
                raise ValueError(f"expected shape {shape}, got {tuple(t.shape)}")
            return t
        n = self.num_envs
        root, thrust, target, ep_ret = prep(root, n, 13), prep(thrust, n, 4), prep(target, n, 3), prep(ep_ret, n)
        check(lib.ozl_set_state(self._h, ptr(root), ptr(thrust), ptr(target), ptr(ep_ret), _stream()))
        torch.cuda.current_stream().synchronize()   # inputs may be temporaries

    def get_params(self):
        n = self.num_envs
        p, f = self._new(n, 8), self._new(n, 2, dtype=torch.int32)
        check(lib.ozl_get_params(self._h, p.data_ptr(), f.data_ptr(), _stream()))
        return p, f

    def set_params(self, params8=None, fault2=None):
        """params8 [N,8] = mass, ixx, iyy, izz, arm, thrust scale, fault effectiveness, yaw_km; fault2 [N,2] = rotor, onset
        (bit 31 of the onset word carries the env's landed flag, so get_params -> set_params round-trips it)."""
        n = self.num_envs
        params7 = params8
        if params7 is not None:
            params7 = params7.to(device=self.device, dtype=torch.float32).contiguous()
            assert tuple(params7.shape) == (n, 8)
        if fault2 is not None:
            fault2 = fault2.to(device=self.device, dtype=torch.int32).contiguous()
            assert tuple(fault2.shape) == (n, 2)
        check(lib.ozl_set_params(self._h, ptr(params7), ptr(fault2), _stream()))
        torch.cuda.current_stream().synchronize()

    def get_rotor_eff(self):
        """fault_mode 2: e_0..e_3 of every env's current episode, [N, 4] float32 CUDA tensor (ozl_get_rotor_eff)."""
        out = self._new(self.num_envs, 4)
        check(lib.ozl_get_rotor_eff(self._h, out.data_ptr(), _stream()), ValueError)
        return out

    def set_rotor_eff(self, eff4):
        """fault_mode 2: replace e_0..e_3 of every env ([N, 4]; the faulted rotors and the onset stay as drawn)."""
        eff4 = eff4.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(eff4.shape) != (self.num_envs, 4):
            raise ValueError(f"expected shape {(self.num_envs, 4)}, got {tuple(eff4.shape)}")
        check(lib.ozl_set_rotor_eff(self._h, eff4.data_ptr(), _stream()), ValueError)
        torch.cuda.current_stream().synchronize()   # the input may be a temporary

    @property
    def step_count(self):
        out = C.c_uint64()
        check(lib.ozl_get_step_count(self._h, C.byref(out), _stream()))
        return out.value

    @step_count.setter
    def step_count(self, v):
        check(lib.ozl_set_step_count(self._h, int(v), _stream()))

    def metrics(self, clear=False, out=None):
        """16-double metrics vector (device tensor).  See include/ouzelum_b200.h for the slots."""
        if out is None:
            out = torch.empty(16, dtype=torch.float64, device=self.device)
        check(lib.ozl_metrics_read(self._h, out.data_ptr(), 1 if clear else 0, _stream()))
        return out


METRIC_NAMES = ("sum_reward", "sum_episode_return", "landed_episodes", None, None, None, None, None,
                "env_steps", "episodes", "sum_episode_length", "timeouts", "crash_dist", "crash_z",
                "fault_active_steps", "resets")
