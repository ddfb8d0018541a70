"""CPU reference of the privileged critic state the step kernels write (ozl_set_states_output; layout OZL_STATE_* in
include/ouzelum_b200.h, device code states_row() in ouzelum_b200/csrc/quad_env.cuh).

The row is a function of the post-step env state, so it is rebuilt here from the CPU oracle's state after each step
(`StatesOracle`) or from the product's own state accessors (`states_from_task`), with the kernel's float32 operations:
IEEE divisions by the cfg values, the observation's own 1/3 scaling for the position, clamp to +-clip_obs."""
import numpy as np
import torch

from oracle.quad_step import QuadStepOracle, compute_observations, div_by_scalar

# slots, restated independently of the header (test_states_cpu.py checks that the two statements agree)
OBS, THRUST, EFF, MASS, THRUST_SCALE, YAW_KM, PROGRESS, POS, WIDTH = 0, 13, 17, 21, 26, 27, 28, 29, 32


def states_row(clean_obs, root, thrust, fault_active, fault_rotor, fault_eff, params7, progress, cfg):
    """[N, 32] float32.  clean_obs: the observation before the sensor-fault model (any clamp is re-applied); params7: mass, ixx,
    iyy, izz, arm, thrust scale, yaw_km; progress: after the step; fault_active: the rotor fault was applied this step."""
    f32 = lambda x: torch.tensor(float(np.float32(x)), dtype=torch.float32)
    n = root.shape[0]
    s = torch.empty(n, WIDTH, dtype=torch.float32)
    s[:, OBS:OBS + 13] = clean_obs
    s[:, THRUST:THRUST + 4] = thrust / f32(cfg["thrust_max"])
    one = torch.ones(n, dtype=torch.float32)
    for i in range(4):
        s[:, EFF + i] = torch.where(fault_active & (fault_rotor == i), fault_eff, one)
    for j, k in enumerate(("mass", "ixx", "iyy", "izz", "arm")):
        s[:, MASS + j] = params7[:, j] / f32(cfg[k])
    s[:, THRUST_SCALE] = params7[:, 5]
    s[:, YAW_KM] = params7[:, 6]
    s[:, PROGRESS] = progress.to(torch.float32) / f32(float(np.float32(cfg["max_episode_length"])))
    s[:, POS:POS + 3] = div_by_scalar(root[:, 0:3], 3)
    clip = float(np.float32(cfg["clip_obs"]))
    return torch.clamp(s, -clip, clip)


class StatesOracle(QuadStepOracle):
    """QuadStepOracle that also produces `states_buf` after every step."""

    def __init__(self, cfg, **kw):
        super().__init__(cfg, **kw)
        self.states_buf = torch.zeros(self.n, WIDTH)

    def step(self, actions, target_in=None, act_mode=0, warmup=None, det_target=None):
        out = super().step(actions, target_in=target_in, act_mode=act_mode, warmup=warmup, det_target=det_target)
        cfg = self.cfg
        prog = self.progress_buf
        # the fault is applied in rotor mode once the post-reset progress (progress after the step - 1) reaches the onset
        active = (prog - 1 >= self.fault_onset) if (cfg["fault_mode"] and act_mode == 0) else torch.zeros(self.n, dtype=torch.bool)
        clip = cfg["clip_obs"]
        clean = torch.clamp(compute_observations(self.root, self.target), -clip, clip)
        self.states_buf = states_row(clean, self.root, self.thrust, active, self.fault_rotor, self.fault_eff, self.params, prog, cfg)
        return out


def states_from_task(env, act_mode=0):
    """The row rebuilt from a task's get_state() / get_params() after a step (CPU tensors); the clean observation is recomputed
    from the root state and the target as the oracle computes it (the kernel's observation before the sensor-fault model)."""
    st = env.sim.get_state()
    p8, f2 = env.sim.get_params()
    cfg = env.native_cfg.to_dict()
    root, thrust = st["root"].cpu(), st["thrust"].cpu()
    p8, f2 = p8.cpu(), f2.cpu().long()
    prog = env.progress_buf.cpu()
    onset = f2[:, 1] & 0x1FFFFFFF
    active = (prog - 1 >= onset) if (cfg["fault_mode"] and act_mode == 0) else torch.zeros(prog.shape[0], dtype=torch.bool)
    params7 = torch.cat([p8[:, 0:6], p8[:, 7:8]], 1)
    clean = torch.clamp(compute_observations(root, st["target"].cpu()), -cfg["clip_obs"], cfg["clip_obs"])
    return states_row(clean, root, thrust, active, f2[:, 0], p8[:, 6], params7, prog, cfg)
