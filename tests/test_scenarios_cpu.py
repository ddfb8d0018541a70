"""Scenario tables (ozl_set_scenarios), without a GPU: the layout the header states, the helpers of ouzelum_b200.scenarios, the CPU
reference's known answers and the kernel instantiations the library carries."""
import math
import os
import re
import subprocess

import pytest
import torch

import scenario_ref as S
from oracle.quad_step import QuadStepOracle, default_cfg


@pytest.fixture(scope="module")
def lib():
    from ouzelum_b200 import _lib           # built by the session's native_library fixture
    return _lib


def test_header_layout_equals_the_reference_layout(lib):
    L = lib.SCENARIO_LAYOUT
    assert lib.SCENARIO_WIDTH == S.WIDTH == 32
    names = ("POS", "QUAT", "LINVEL", "ANGVEL", "TARGET", "FAULT_ROTOR", "FAULT_ONSET", "FAULT_EFF", "MASS", "IXX", "IYY", "IZZ",
             "ARM", "THRUST_SCALE", "YAW_KM", "RESERVED")
    assert [L["OZL_SCN_" + k] for k in names] == [S.POS, S.QUAT, S.LINVEL, S.ANGVEL, S.TARGET, S.ROTOR, S.ONSET, S.EFF, S.MASS, S.IXX,
                                                  S.IYY, S.IZZ, S.ARM, S.THRUST_SCALE, S.YAW_KM, S.RESERVED]
    assert (S.POS, S.QUAT, S.LINVEL, S.ANGVEL, S.TARGET, S.MASS, S.RESERVED) == (0, 3, 7, 10, 13, 19, 26)


def test_empty_and_fault_grid(lib):
    from ouzelum_b200 import scenarios
    e = scenarios.empty(5)
    assert e.shape == (5, 32) and e.dtype == torch.float32 and torch.isnan(e).all()
    g = scenarios.fault_grid(10, rotors=[0, 2], onsets=[0, 300], effectiveness=[0.1])
    assert g.shape == (10, 32)
    combos = [(0, 0, 0.1), (0, 300, 0.1), (2, 0, 0.1), (2, 300, 0.1)]
    for i in range(10):
        assert g[i, 16:19].tolist() == pytest.approx(list(combos[i % 4]))
    assert torch.isnan(g[:, :16]).all() and torch.isnan(g[:, 19:]).all()
    assert g[0, 18].item() == torch.tensor(0.1, dtype=torch.float32).item()
    with pytest.raises(ValueError):
        scenarios.fault_grid(4, [], [0], [0.5])


def _actions(n, t):
    g = torch.Generator().manual_seed(500 + t)
    return (torch.rand(n, 4, generator=g) * 2 - 1) * 0.3


ROUGH = dict(seed=7, fault_mode=1, dr_enable=1, pomdp_mode=3, pomdp_prob=0.3, noise_sigma=0.15, max_episode_length=40,
             target_period=7, lin_drag=0.05, yaw_km=0.016)


def test_all_nan_rows_are_the_oracle():
    n = 48
    a, b = QuadStepOracle(default_cfg(n, **ROUGH)), S.ScenarioOracle(default_cfg(n, **ROUGH), S.empty(n))
    for t in range(60):
        act = _actions(n, t)
        a.step(act)
        b.step(act)
        for k in ("obs_buf", "rew_buf", "reset_buf", "progress_buf", "root", "target", "params", "fault_onset", "fault_eff"):
            assert torch.equal(getattr(a, k), getattr(b, k)), (t, k)


def test_pinned_groups_hold_at_every_reset_and_resample():
    n = 6
    cfg = default_cfg(n, **ROUGH)
    rows = S.empty(n)
    rows[0, 0:13] = torch.tensor([0.5, -0.5, 2.0, 0, 0, 0.6, 0.8, 0.1, 0.2, -0.3, 0.0, 0.5, -0.5])
    rows[0, 13:16] = torch.tensor([1.0, 2.0, 1.5])
    rows[0, 16:19] = torch.tensor([2.0, 5.0, 0.25])
    rows[0, 19:26] = torch.tensor([2.5, 0.03, 0.031, 0.05, 0.2, 0.9, 0.02])
    rows[1, 16:19] = torch.tensor([-1.0, 0.0, 0.5])         # no fault this episode
    rows[2, 19] = 3.0                                        # mass only
    ora = S.ScenarioOracle(cfg, rows)
    ora.step(torch.zeros(n, 4))                              # step 0 resets every env
    assert ora.params[0].tolist() == rows[0, 19:26].tolist()
    assert (ora.fault_rotor[0].item(), ora.fault_onset[0].item(), ora.fault_eff[0].item()) == (2, 5, 0.25)
    assert (ora.fault_rotor[1].item(), ora.fault_onset[1].item(), ora.fault_eff[1].item()) == (0, S.FAULT_NEVER, 0.5)
    assert ora.params[2, 0].item() == 3.0 and ora.params[2, 1].item() != 3.0
    resets = 0
    for t in range(1, 90):                                   # target_period 7: many periodic re-samples
        ora.step(_actions(n, t))
        assert ora.target[0].tolist() == [1.0, 2.0, 1.5], t
        resets += int(ora.reset_buf[0])
    assert resets > 0
    # the states row shows the pinned effectiveness once the fault is active (onset 5) and the pinned mass ratio
    ora2 = S.ScenarioOracle(cfg, rows)
    for t in range(7):
        ora2.step(torch.zeros(n, 4))
    assert ora2.states_buf[0, 17 + 2].item() == 0.25
    assert ora2.states_buf[0, 21].item() == (torch.tensor(2.5) / torch.tensor(cfg["mass"], dtype=torch.float32)).item()


def test_fully_pinned_env_does_not_depend_on_the_seed():
    n = 8
    rows = S.mixed_rows(n, default_cfg(n, **ROUGH), seed=3)
    kw = dict(ROUGH, pomdp_mode=0)
    a, b = S.ScenarioOracle(default_cfg(n, **dict(kw, seed=1)), rows), S.ScenarioOracle(default_cfg(n, **dict(kw, seed=2)), rows)
    full = torch.arange(n) % 3 == 0
    for t in range(100):
        act = _actions(n, t)
        a.step(act)
        b.step(act)
        assert torch.equal(a.root[full], b.root[full]) and torch.equal(a.rew_buf[full], b.rew_buf[full]), t
    assert not torch.equal(a.root[~full], b.root[~full])


def _res_usage(lib):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    out = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-res-usage", lib.LIB_PATH],
                         capture_output=True, text=True).stdout
    return {m.group(1): dict((k, int(v)) for k, v in re.findall(r"(\w+):(\d+)", m.group(2)))
            for m in re.finditer(r"Function (\S+):\s*\n\s*(REG:.*)", out)}


def test_scenario_kernels_keep_the_occupancy_of_the_kernels_without_a_table(lib):
    """Every step kernel has a scenario twin; the twin uses no local memory and fits the same CTAs per SM (generic 7 x 128
    threads, TMA 5; 228 KB of shared memory per SM including the 1 KB the driver reserves per CTA)."""
    ru = _res_usage(lib)
    plain, scn = {}, {}
    for name, r in ru.items():
        m = re.match(r"_ZN3ozl(16quad_step_kernel|20quad_step_scn_kernel|20quad_step_tma_kernel|24quad_step_tma_scn_kernel)I(\w*?)EEv",
                     name)
        if m:
            (scn if "scn" in m.group(1) else plain)[("tma" if "tma" in m.group(1) else "gen", m.group(2))] = r
    assert len(plain) == 8 and sorted(plain) == sorted(scn), (sorted(plain), sorted(scn))
    for key, r in scn.items():
        ctas = 5 if key[0] == "tma" else 7
        assert r["LOCAL"] == 0 and r["STACK"] <= plain[key]["STACK"], (key, r, plain[key])
        assert r["REG"] * 128 * ctas <= 65536 and (r["SHARED"] + 1024) * ctas <= 228 * 1024, (key, r)
        assert r["SHARED"] == plain[key]["SHARED"], key


def test_set_scenarios_needs_a_handle(lib):
    L = lib.lib
    assert L.ozl_set_scenarios(None, None, 32, None) != 0 and "env is NULL" in L.ozl_last_error().decode()
    assert math.isnan(float(S.empty(1)[0, 31]))
