"""CPU reference of the episode log (ozl_set_episode_log; record layout OZL_EPLOG_* in include/ouzelum_b200.h, device code
log_episode() in ouzelum_b200/csrc/quad_step.cu): the record of every env whose episode ends in a step, built from the oracle's state
after that step.

`with_episode_log(cls)` puts the recording in front of an oracle class (QuadStepOracle or one of the test subclasses in
scenario_ref / multi_fault_ref / metrics_ref); oracle/ stays unchanged.  `log_rows()` is the record set as uint32 bits [k, 32], sorted
by (step, env) -- the order the kernels write them in is not deterministic, their contents are."""
import numpy as np
import torch

from oracle.quad_step import QuadStepOracle

# slots, restated independently of the header (test_episode_log_cpu.py checks that the two statements agree)
ENV, LENGTH, STEP, RETURN, FLAGS, ONSET, DIST, EFF = 0, 1, 2, 4, 5, 6, 7, 8
MASS, POS, LINVEL, TARGET, RESERVED, WIDTH = 12, 19, 22, 25, 28, 32
TIMEOUT, CRASH_DIST, CRASH_Z, LANDED, FAULT_ACTIVE = 1, 2, 4, 8, 16        # bits of FLAGS
FAULT_NEVER = 0x1FFFFFFF


def f32_bits(x):
    return np.asarray(x, dtype=np.float32).view(np.uint32)


def dist32(target, pos):
    """Distance to the target, float32 as the kernel computes it ((dx^2 + dy^2) + dz^2, correctly rounded sqrt)."""
    d = (target - pos).to(torch.float32).numpy()
    return np.sqrt(((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]).astype(np.float32))


class EpisodeLogMixin:
    """Records, after every `step`, one row per env whose episode ended in it."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self._rows = []

    def step(self, actions, target_in=None, act_mode=0, warmup=None, det_target=None):
        t = self.step_count
        out = super().step(actions, target_in=target_in, act_mode=act_mode, warmup=warmup, det_target=det_target)
        done = (self.reset_buf != 0).numpy()
        if not done.any():
            return out
        cfg = self.cfg
        prog = self.progress_buf
        mode = cfg["fault_mode"]
        active = ((prog - 1 >= self.fault_onset) if (mode and act_mode == 0) else torch.zeros(self.n, dtype=torch.bool)).numpy()
        onset = self.fault_onset.numpy().astype(np.int64)
        if mode == 2:
            eff = self.rotor_eff.numpy().astype(np.float32)                 # as drawn, not ramped
        else:
            eff = np.ones((self.n, 4), dtype=np.float32)
            if mode == 1:
                hit = onset != FAULT_NEVER
                rotor = self.fault_rotor.numpy()
                eff[hit, rotor[hit]] = self.fault_eff.numpy().astype(np.float32)[hit]
        root = self.root.to(torch.float32)
        dist = dist32(self.target, root[:, 0:3])
        flags = (self.timeout_buf.numpy().astype(np.uint32) * TIMEOUT
                 | (dist > np.float32(cfg["die_dist"])).astype(np.uint32) * CRASH_DIST
                 | (root[:, 2].numpy() < np.float32(cfg["die_z"])).astype(np.uint32) * CRASH_Z
                 | self.landed.numpy().astype(np.uint32) * LANDED
                 | active.astype(np.uint32) * FAULT_ACTIVE)
        r = np.zeros((self.n, WIDTH), dtype=np.uint32)
        r[:, ENV] = self.env_ids.astype(np.uint32)
        r[:, LENGTH] = prog.numpy().astype(np.int64).astype(np.uint32)
        r[:, STEP] = np.uint32(t & 0xFFFFFFFF)
        r[:, STEP + 1] = np.uint32(t >> 32)
        r[:, RETURN] = f32_bits(self.returned_ep_ret.to(torch.float32).numpy())
        r[:, FLAGS] = flags
        r[:, ONSET] = np.where(onset == FAULT_NEVER, -1, onset).astype(np.int64).astype(np.uint32)
        r[:, DIST] = f32_bits(dist)
        r[:, EFF:EFF + 4] = f32_bits(eff)
        r[:, MASS:MASS + 7] = f32_bits(self.params.to(torch.float32).numpy())
        r[:, POS:POS + 3] = f32_bits(root[:, 0:3].numpy())
        r[:, LINVEL:LINVEL + 3] = f32_bits(root[:, 7:10].numpy())
        r[:, TARGET:TARGET + 3] = f32_bits(self.target.to(torch.float32).numpy())
        self._rows.append(r[done])
        return out

    def log_rows(self):
        """Every record so far, uint32 [k, WIDTH], sorted by (step, env)."""
        return sort_rows(np.concatenate(self._rows) if self._rows else np.zeros((0, WIDTH), dtype=np.uint32))

    def clear_log(self):
        self._rows = []


def sort_rows(bits):
    """uint32 [k, WIDTH] records in (step, env) order."""
    bits = np.asarray(bits).view(np.uint32).reshape(-1, WIDTH)
    step = bits[:, STEP].astype(np.uint64) | (bits[:, STEP + 1].astype(np.uint64) << np.uint64(32))
    return bits[np.lexsort((bits[:, ENV], step))]


def tallies(bits, last_step=None):
    """What the metrics vector counts of these records: {slot: value} for slots 9 (episodes), 10 (sum of lengths), 11 (time-outs),
    12 / 13 (the crash causes), 2 (landed episodes: the metrics count one at the NEXT step's reset, so only records of steps
    before `last_step` count), and the float32 returns (slot 1's terms)."""
    bits = np.asarray(bits, dtype=np.uint32).reshape(-1, WIDTH)
    f = bits[:, FLAGS]
    landed = (f & LANDED) != 0
    if last_step is not None:
        landed &= bits[:, STEP] < np.uint32(last_step)
    return {9: len(bits), 10: int(bits[:, LENGTH].astype(np.int64).sum()), 11: int(((f & TIMEOUT) != 0).sum()),
            12: int(((f & CRASH_DIST) != 0).sum()), 13: int(((f & CRASH_Z) != 0).sum()), 2: int(landed.sum()),
            "returns": bits[:, RETURN].view(np.float32).astype(np.float64)}


def with_episode_log(cls=QuadStepOracle):
    return type("EpisodeLog" + cls.__name__, (EpisodeLogMixin, cls), {})
