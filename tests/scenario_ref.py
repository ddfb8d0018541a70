"""CPU reference of the scenario table (ozl_set_scenarios; layout OZL_SCN_* in include/ouzelum_b200.h, device code scn_target() /
scn_respawn() in ouzelum_b200/csrc/quad_env.cuh): the oracle's step with the rows laid over its reset draws.

The oracle draws the reset conditions and then assigns them to its state attributes (target, root, fault_rotor / _onset / _eff,
params) before it computes the actuation and the physics.  `ScenarioOracle` leaves oracle/ untouched: it turns those attributes
into properties and, during the reset phase of a step, lays the set groups of each row over the first assignment of each one --
exactly where the kernel overwrites the draws.  It derives from `StatesOracle`, so the privileged state row follows too."""
import math

import torch

from states_ref import StatesOracle

# slots, restated independently of the header (test_scenarios_cpu.py checks that the two statements agree)
POS, QUAT, LINVEL, ANGVEL, TARGET, ROTOR, ONSET, EFF = 0, 3, 7, 10, 13, 16, 17, 18
MASS, IXX, IYY, IZZ, ARM, THRUST_SCALE, YAW_KM, RESERVED, WIDTH = 19, 20, 21, 22, 23, 24, 25, 26, 32
ROOT_GROUPS = ((POS, 3), (QUAT, 4), (LINVEL, 3), (ANGVEL, 3))      # slots 0-12 are root13
FAULT_NEVER = 0x1FFFFFFF


def empty(n):
    return torch.full((n, WIDTH), math.nan, dtype=torch.float32)


class ScenarioOracle(StatesOracle):
    """StatesOracle whose resets apply `rows` ([N, 32] float32, NaN groups keep the draw)."""

    _LAID = ("target", "root", "fault_rotor", "fault_onset", "fault_eff", "params")

    def __init__(self, cfg, rows, **kw):
        self._pending = ()
        super().__init__(cfg, **kw)
        self.rows = rows.to(torch.float32).clone()

    def _set(self, slot):
        return ~torch.isnan(self.rows[:, slot])

    def _lay(self, name, v):
        r, rst = self.rows, self._rst
        if name == "target":                     # at every re-sample: the reset and the periodic ones
            m = self._resample & self._set(TARGET)
            return torch.where(m[:, None], r[:, TARGET:TARGET + 3], v)
        if name == "root":
            v = v.clone()
            for first, k in ROOT_GROUPS:
                m = rst & self._set(first)
                v[:, first:first + k] = torch.where(m[:, None], r[:, first:first + k], v[:, first:first + k])
            return v
        if name == "params":                     # mass, ixx, iyy, izz, arm, thrust scale, yaw_km
            v = v.clone()
            for j in range(7):
                m = rst & self._set(MASS + j)
                v[:, j] = torch.where(m, r[:, MASS + j], v[:, j])
            return v
        m = rst & self._set(ROTOR)
        none = r[:, ROTOR] < 0                   # rotor -1: no fault this episode
        if name == "fault_rotor":
            return torch.where(m, torch.where(none, 0.0, r[:, ROTOR]).to(torch.int64), v)
        if name == "fault_onset":
            return torch.where(m, torch.where(none, FAULT_NEVER, r[:, ONSET].to(torch.int64)), v)
        return torch.where(m, r[:, EFF], v)       # fault_eff

    def step(self, actions, target_in=None, act_mode=0, warmup=None, det_target=None):
        cfg = self.cfg
        self._rst = self.reset_buf != 0
        self._resample = ((self.progress_buf % cfg["target_period"]) == 0) | self._rst
        if cfg.get("target_fixed", 0):
            self._resample = torch.zeros_like(self._rst)
        pending = set(self._LAID)
        if not cfg["dr_enable"]:                 # no draw assigns the body parameters: lay the rows over the kept values now
            self.params = self._lay("params", self.params)
            pending.discard("params")
        self._pending = pending
        try:
            return super().step(actions, target_in=target_in, act_mode=act_mode, warmup=warmup, det_target=det_target)
        finally:
            self._pending = ()


def _laid_property(name):
    def get(self):
        return self.__dict__["_" + name]

    def put(self, v):
        if name in self._pending:
            self._pending.discard(name)
            v = self._lay(name, v)
        self.__dict__["_" + name] = v
    return property(get, put)


for _name in ScenarioOracle._LAID:
    setattr(ScenarioOracle, _name, _laid_property(_name))


def mixed_rows(n, cfg, seed=0):
    """A mixed table for the equivalence tests: every 3rd env fully pinned, every 3rd + 1 partly pinned (position, fault, mass,
    thrust scale), the rest NaN.  Groups the cfg would refuse (target with target_fixed, fault without fault_mode) stay NaN."""
    g = torch.Generator().manual_seed(seed)
    u = lambda *s: torch.rand(*s, generator=g, dtype=torch.float64)
    rows = empty(n)
    full, part = torch.arange(n) % 3 == 0, torch.arange(n) % 3 == 1
    q = torch.randn(n, 4, generator=g, dtype=torch.float64) * torch.tensor([0.1, 0.1, 0.1, 1.0], dtype=torch.float64)
    q = (q / q.norm(dim=1, keepdim=True)).float()
    pos = torch.stack([u(n) * 3 - 1.5, u(n) * 3 - 1.5, u(n) * 1.5 + 0.8], 1).float()
    nominal = torch.tensor([cfg["mass"], cfg["ixx"], cfg["iyy"], cfg["izz"], cfg["arm"], 1.0, 0.01], dtype=torch.float64)
    body = (nominal * (0.8 + 0.4 * u(n, 7))).float()
    fault = torch.stack([torch.randint(-1, 4, (n,), generator=g).double(), torch.randint(0, 30, (n,), generator=g).double(),
                         u(n)], 1).float()
    rows[full, POS:POS + 3] = pos[full]
    rows[full, QUAT:QUAT + 4] = q[full]
    rows[full, LINVEL:LINVEL + 3] = (u(n, 3)[full] - 0.5).float()
    rows[full, ANGVEL:ANGVEL + 3] = (u(n, 3)[full] - 0.5).float()
    if not cfg.get("target_fixed", 0):
        rows[full, TARGET:TARGET + 3] = torch.stack([u(n) * 4 - 2, u(n) * 4 - 2, u(n) + 1], 1).float()[full]
    rows[full, MASS:YAW_KM + 1] = body[full]
    rows[part, POS:POS + 3] = pos[part]
    rows[part, MASS] = body[part, 0]
    rows[part, THRUST_SCALE] = body[part, 5]
    if cfg["fault_mode"]:
        rows[full | part, ROTOR:EFF + 1] = fault[full | part]
    return rows
