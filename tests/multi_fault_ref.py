"""CPU reference of rotorFault mode "multi" (cfg.fault_mode 2; the law is stated in include/ouzelum_b200.h, "Rotor faults, mode 2";
device code rfault_draw() / rfault_factors() / scn_rfault() in ouzelum_b200/csrc/quad_env.cuh).

`MultiFaultOracle` derives from `ScenarioOracle` (so the states row and scenario tables follow) and leaves oracle/ untouched: it runs
the parent step with fault_mode 0 -- no mode-1 draw, no single-rotor fault --, draws the mode-2 conditions of the resetting envs
itself, multiplies the four rotor forces by a_j right before the integrator (`_simulate`, where the kernel applies them too) and
restores fault_mode 2 afterwards, so that the metrics tally (metrics_ref.with_metrics) sees the fault as active from the onset."""
import itertools

import numpy as np
import torch

import scenario_ref as S
from oracle import philox as px
from oracle.quad_step import fma

# restated independently of the device code (test_multi_fault_cpu.py checks them against the header and philox.cuh)
P_RFAULT = 7
RONSET, REFF = 26, 27
FAULT_NEVER = 0x1FFFFFFF
PERMS = list(itertools.permutations(range(4)))          # the 24 permutations of {0,1,2,3}, lexicographic


def f32(x):
    return torch.tensor(float(np.float32(x)), dtype=torch.float32)


def reset_draw(cfg, env_ids, step):
    """The conditions a reset at `step` draws: onset (int64 [n], FAULT_NEVER when k = 0), e (float32 [n, 4]), k and the
    permutation index (int64 [n]).  Words r0..r2 of P_FAULT and w0..w3 of P_RFAULT, keyed by (seed, global env id, step)."""
    seed = cfg.get("seed", 0)
    r0, r1, r2, _ = px.draw(seed, env_ids, step, px.P_FAULT)
    w = px.draw(seed, env_ids, step, P_RFAULT)
    lo, hi = int(cfg.get("fault_rotors_lo", 1)), int(cfg.get("fault_rotors_hi", 1))
    k = lo + px.mulhi(r2, hi - lo + 1)                                   # k = lo + umulhi(r2, hi - lo + 1)
    perm = px.mulhi(r0, 24)                                              # permutation umulhi(r0, 24)
    onset = np.where(k > 0, px.mulhi(r1, cfg["max_episode_length"]), FAULT_NEVER)
    e = torch.ones(len(k), 4, dtype=torch.float32)
    lo_e, rng = f32(cfg["fault_eff_lo"]), f32(cfg["fault_eff_range"])
    for j in range(4):
        faulted = torch.tensor([j in PERMS[p][:kk] for p, kk in zip(perm.tolist(), k.tolist())], dtype=torch.bool)
        u = torch.from_numpy(px.u01(w[j]))
        e[:, j] = torch.where(faulted, lo_e + rng * u, torch.ones(()))   # e_j = fault_eff_lo + fault_eff_range * u01(w_j)
    return torch.from_numpy(onset.astype(np.int64)), e, torch.from_numpy(k), torch.from_numpy(perm)


def ramp_factor(e, d, ramp):
    """One rotor, literally as the header states it: a_j = e_j if ramp <= 1 or d + 1 >= ramp, else
    fmaf((float)(d + 1) * inv_ramp, e_j - 1.0f, 1.0f) with inv_ramp = (float)(1.0 / ramp).  e: float32, d >= 0: int."""
    e = np.float32(e)
    if ramp <= 1 or d + 1 >= ramp:
        return e
    inv_ramp = np.float32(1.0 / ramp)
    x = np.float32(np.float32(d + 1) * inv_ramp)
    return np.float32(fma(torch.tensor(x), torch.tensor(np.float32(e - np.float32(1.0))), 1.0).item())


def factors(e, onset, prog, ramp):
    """a [n, 4] and `active` [n] at post-reset progress `prog` (the vectorised ramp_factor; 1 before the onset)."""
    active = prog >= onset
    d = prog - onset
    a = e.clone()
    if ramp > 1:
        part = active & (d + 1 < ramp)
        x = torch.where(part, d + 1, 0).to(torch.float32) * f32(1.0 / ramp)
        a = torch.where(part[:, None], fma(x[:, None].expand(-1, 4).contiguous(), e - 1.0, 1.0), e)
    return torch.where(active[:, None], a, torch.ones(())), active


def lay_rows(rows, onset, e):
    """The rotor-faults group of scenario rows over drawn conditions: pinned rows give their onset / e, four 1s mean no fault."""
    pinned = ~torch.isnan(rows[:, RONSET])
    pe = rows[:, REFF:REFF + 4]
    none = (pe == 1.0).all(1)
    onset = torch.where(pinned, torch.where(none, FAULT_NEVER, torch.nan_to_num(rows[:, RONSET]).long()), onset)
    return onset, torch.where(pinned[:, None], pe, e)


class MultiFaultOracle(S.ScenarioOracle):
    """ScenarioOracle of a fault_mode 2 cfg: `rotor_eff` [n, 4] holds e_0..e_3, `fault_onset` the onset, `applied_eff` the a_j
    of the last step (what OZL_STATE_EFF reports)."""

    def __init__(self, cfg, rows=None, **kw):
        n = int(cfg["num_envs"])
        super().__init__(cfg, S.empty(n) if rows is None else rows, **kw)
        assert self.cfg["fault_mode"] == 2
        self.rotor_eff = torch.ones(n, 4, dtype=torch.float32)
        self.applied_eff = torch.ones(n, 4, dtype=torch.float32)
        self._a = None

    def pending_reset(self):
        """(onset, e) every env would get if it reset at the current step (what ozl_apply_resets writes)."""
        onset, e, _, _ = reset_draw(self.cfg, self.env_ids, self.step_count)
        return lay_rows(self.rows, onset, e)

    def step(self, actions, target_in=None, act_mode=0, warmup=None, det_target=None):
        cfg = self.cfg
        rst = self.reset_buf != 0
        onset, e = self.pending_reset()
        self.fault_onset = torch.where(rst, onset, self.fault_onset)
        self.rotor_eff = torch.where(rst[:, None], e, self.rotor_eff)
        prog = torch.where(rst, torch.zeros_like(self.progress_buf), self.progress_buf)
        a, _ = factors(self.rotor_eff, self.fault_onset, prog, int(cfg.get("fault_ramp_steps", 0)))
        self.applied_eff = a if act_mode == 0 else torch.ones_like(a)
        self._a = a if act_mode == 0 else None
        cfg["fault_mode"] = 0
        try:
            out = super().step(actions, target_in=target_in, act_mode=act_mode, warmup=warmup, det_target=det_target)
        finally:
            cfg["fault_mode"] = 2
            self._a = None
        clip = float(np.float32(cfg["clip_obs"]))
        self.states_buf[:, 17:21] = torch.clamp(self.applied_eff, -clip, clip)
        return out

    def _simulate(self, force, wrench=None, body_force=None):
        if force is not None and self._a is not None:
            force = force * self._a                  # a_j = 1 exactly for a healthy rotor and before the onset
        return super()._simulate(force, wrench=wrench, body_force=body_force)
