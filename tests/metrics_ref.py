"""CPU reference of the episode-metrics vector (ozl_metrics_read; slots in include/ouzelum_b200.h and quad_io.cuh's
block_epilogue): what every step of the oracle adds to each of the 16 slots.

Counts are exact Python ints.  For the two float slots the reference keeps every float32 term -- the reward of every env, the
episode return of every env whose episode ended -- and its value is `math.fsum` over them: the exact sum, rounded once.  The
kernels add the same exactly representable terms in float64 in some tree order, so a device sum of m terms may differ from the
exact sum by at most (m - 1) * 2^-53 * sum |terms| (`bound`), the worst case of float64 summation in any order.

`with_metrics(cls)` adds the tallies to the oracle class `cls` (QuadStepOracle or one of its test subclasses); oracle/ stays
unchanged.  `QuadStepOracle.load` does not touch the tallies, so they keep accumulating over steps taken from reloaded state."""
import math

import numpy as np
import torch

from oracle.quad_step import QuadStepOracle

# slot layout, restated from the header
SUM_REWARD, SUM_RETURN, LANDED = 0, 1, 2
ENV_STEPS, EPISODES, SUM_LENGTH, TIMEOUTS, CRASH_DIST, CRASH_Z, FAULT_STEPS, RESETS = 8, 9, 10, 11, 12, 13, 14, 15
FLOAT_SLOTS = (SUM_REWARD, SUM_RETURN)
COUNT_SLOTS = (LANDED,) + tuple(range(3, 16))            # 3..7 are reserved: always 0


class MetricsMixin:
    """Records the metrics contribution of every `step`; put it in front of an oracle class (see `with_metrics`)."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.clear_metrics()

    def clear_metrics(self):
        self.counts = [0] * 16
        self.terms = {SUM_REWARD: [], SUM_RETURN: []}

    def step(self, actions, target_in=None, act_mode=0, warmup=None, det_target=None):
        rst = (self.reset_buf != 0).clone()                  # resets this step applies
        out = super().step(actions, target_in=target_in, act_mode=act_mode, warmup=warmup, det_target=det_target)
        cfg = self.cfg
        done = self.reset_buf != 0
        prog = self.progress_buf                              # after the step: the length of an episode that ended
        # the rotor fault acts from the post-reset progress (= progress after the step - 1) on; never under wrench actuation
        if cfg["fault_mode"] and act_mode == 0:
            fault = prog - 1 >= self.fault_onset
        else:
            fault = torch.zeros(self.n, dtype=torch.bool)
        c = self.counts
        c[LANDED] += int(self._landed_episode.sum())
        c[ENV_STEPS] += self.n
        c[EPISODES] += int(done.sum())
        c[SUM_LENGTH] += int(prog[done].sum())
        c[TIMEOUTS] += int(self.timeout_buf.sum())
        c[CRASH_DIST] += int((self._dist32() > np.float32(cfg["die_dist"])).sum())
        c[CRASH_Z] += int((self.root[:, 2] < np.float32(cfg["die_z"])).sum())
        c[FAULT_STEPS] += int(fault.sum())
        c[RESETS] += int(rst.sum())
        self.terms[SUM_REWARD].append(self.rew_buf.numpy().astype(np.float32).copy())
        self.terms[SUM_RETURN].append(self.returned_ep_ret[done].numpy().astype(np.float32).copy())
        return out

    def _dist32(self):
        """Distance to the target after the step, float32 as the kernel computes it ((dx^2 + dy^2) + dz^2, correctly rounded sqrt)."""
        d = (self.target - self.root[:, 0:3]).to(torch.float32).numpy()
        s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        return np.sqrt(s.astype(np.float32))

    # ---- the reference vector and the tolerance of its float slots
    def _flat(self, slot):
        t = self.terms[slot]
        return np.concatenate(t).astype(np.float64) if t else np.zeros(0)

    def vector(self):
        """16 float64: slots 0-1 the exact sums rounded once, every other slot an exact count (3..7: 0)."""
        v = np.array([float(x) for x in self.counts], dtype=np.float64)
        for s in FLOAT_SLOTS:
            v[s] = math.fsum(self._flat(s).tolist())
        return v

    def bound(self, slot):
        """(m - 1) * 2^-53 * sum |terms|: the most a float64 sum of the slot's m terms, in any order, may differ from the exact sum."""
        t = self._flat(slot)
        return max(len(t) - 1, 0) * 2.0 ** -53 * math.fsum(np.abs(t).tolist())

    def n_terms(self, slot):
        return sum(len(t) for t in self.terms[slot])


def with_metrics(cls=QuadStepOracle):
    return type("Metrics" + cls.__name__, (MetricsMixin, cls), {})


MetricsOracle = with_metrics(QuadStepOracle)


def assert_metrics(got, ref, tag=""):
    """The comparison rule: slots 2-15 equal to the reference (3-7 zero), slots 0-1 within `ref.bound`."""
    got = np.asarray(got.cpu() if isinstance(got, torch.Tensor) else got, dtype=np.float64)
    want = ref.vector()
    bad = [s for s in COUNT_SLOTS if got[s] != want[s]]
    assert not bad, f"{tag}: count slots {bad} differ: got {[got[s] for s in bad]}, reference {[want[s] for s in bad]}"
    for s in FLOAT_SLOTS:
        err, tol = abs(got[s] - want[s]), ref.bound(s)
        assert err <= tol, f"{tag}: slot {s} = {got[s]!r}, exact {want[s]!r}: |error| {err:.3e} > bound {tol:.3e}"
