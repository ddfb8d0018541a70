"""Episode log (ozl_set_episode_log) without a GPU: the header and binding layout, the refusals that need no device, the CPU
reference's records against the metrics reference's tallies, and the resources of the log kernel twins."""
import ctypes as C
import math
import re

import numpy as np
import pytest
import torch

import episode_log_ref as E
import multi_fault_ref as M
from metrics_ref import with_metrics
from oracle.quad_step import QuadStepOracle, default_cfg
from test_multi_fault_cpu import _ptxas_spills, _res_usage


@pytest.fixture(scope="module")
def lib():
    from ouzelum_b200 import _lib
    return _lib


def test_header_and_binding_layout(lib):
    L = lib.EPLOG_LAYOUT
    assert lib.OZL_ABI_VERSION == 7 and lib.lib.ozl_abi_version() == 7
    assert lib.lib.ozl_cfg_size() == C.sizeof(lib.OzlCfg) == 408            # registered, not configured: ozl_cfg is unchanged
    want = {"OZL_EPLOG_ENV": E.ENV, "OZL_EPLOG_LENGTH": E.LENGTH, "OZL_EPLOG_STEP": E.STEP, "OZL_EPLOG_RETURN": E.RETURN,
            "OZL_EPLOG_FLAGS": E.FLAGS, "OZL_EPLOG_ONSET": E.ONSET, "OZL_EPLOG_DIST": E.DIST, "OZL_EPLOG_EFF": E.EFF,
            "OZL_EPLOG_MASS": E.MASS, "OZL_EPLOG_IXX": 13, "OZL_EPLOG_IYY": 14, "OZL_EPLOG_IZZ": 15, "OZL_EPLOG_ARM": 16,
            "OZL_EPLOG_THRUST_SCALE": 17, "OZL_EPLOG_YAW_KM": 18, "OZL_EPLOG_POS": E.POS, "OZL_EPLOG_LINVEL": E.LINVEL,
            "OZL_EPLOG_TARGET": E.TARGET, "OZL_EPLOG_RESERVED": E.RESERVED, "OZL_EPLOG_WIDTH": E.WIDTH}
    assert L == want and lib.EPLOG_WIDTH == 32
    # the body parameters in the scenario row's order (params8 without the mode-1 effectiveness)
    S = lib.SCENARIO_LAYOUT
    assert [L[k.replace("SCN", "EPLOG")] - L["OZL_EPLOG_MASS"] for k in
            ("OZL_SCN_MASS", "OZL_SCN_IXX", "OZL_SCN_IYY", "OZL_SCN_IZZ", "OZL_SCN_ARM", "OZL_SCN_THRUST_SCALE", "OZL_SCN_YAW_KM")] == \
        [S[k] - S["OZL_SCN_MASS"] for k in ("OZL_SCN_MASS", "OZL_SCN_IXX", "OZL_SCN_IYY", "OZL_SCN_IZZ", "OZL_SCN_ARM",
                                             "OZL_SCN_THRUST_SCALE", "OZL_SCN_YAW_KM")]
    assert not any(k.startswith("OZL_EPLOG") for k in list(lib.SCENARIO_LAYOUT) + list(lib.STATES_LAYOUT))
    assert lib._SIGS["ozl_set_episode_log"] == (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32])


def test_refusals_without_a_device(lib):
    buf = (C.c_float * 64)()
    head = C.c_uint64(0)
    assert lib.lib.ozl_set_episode_log(None, buf, 2, C.byref(head), 32) != 0 and "env is NULL" in lib.last_error()
    from ouzelum_b200.tasks.ekf_lee_landed import EKFLeeLanded
    from ouzelum_b200.tasks.landing import Landed, Landing, Lando
    from ouzelum_b200.tasks.lee_landed import LeeLanded
    from ouzelum_b200.tasks.ouzelum import Ouzelum
    from ouzelum_b200.tasks.quadcopter import Quadcopter
    assert all(c.supports_episode_log for c in (Ouzelum, Lando, Landing, Landed, LeeLanded))
    assert not EKFLeeLanded.supports_episode_log and not Quadcopter.supports_episode_log
    for cls in (EKFLeeLanded, Quadcopter):                  # refused before anything touches a device
        with pytest.raises(ValueError, match="episode log is not supported"):
            cls.__new__(cls).enable_episode_log(16)


def test_decode_of_reference_rows():
    """decode_episode_records reads back what the reference writes (no device: CPU tensors)."""
    from ouzelum_b200.tasks.ouzelum import decode_episode_records
    cfg = default_cfg(64, seed=4, max_episode_length=32, fault_mode=1, dr_enable=1, env_id_base=7)
    ora = E.with_episode_log(QuadStepOracle)(cfg)
    g = torch.Generator().manual_seed(1)
    for _ in range(40):
        ora.step(torch.rand(64, 4, generator=g) * 2 - 1)
    bits = ora.log_rows()
    d = decode_episode_records(torch.from_numpy(bits.view(np.float32)[::-1].copy()))
    assert torch.equal(d["env"], torch.from_numpy(bits[:, E.ENV].astype(np.int64)))
    assert torch.equal(d["step"], torch.from_numpy(bits[:, E.STEP].astype(np.int64)))
    assert torch.equal(d["length"], torch.from_numpy(bits[:, E.LENGTH].astype(np.int64)))
    assert torch.equal(d["params"], torch.from_numpy(bits[:, E.MASS:E.MASS + 7].view(np.float32)))
    assert int(d["timeout"].sum()) == int(((bits[:, E.FLAGS] & E.TIMEOUT) != 0).sum()) > 0
    assert int((d["onset"] >= 0).sum()) == len(bits) > 0                 # mode 1 schedules a fault in every episode


def test_decode_orders_steps_beyond_int32():
    """(step, env) order holds for step indices of 2^31 and more, where a packed 64-bit key would overflow."""
    from ouzelum_b200.tasks.ouzelum import decode_episode_records
    steps = [(1 << 33) + 5, 3, (1 << 31) + 1, (1 << 33) + 5, (1 << 31)]
    envs = [7, 0xFFFFFFFF, 2, 1, 0xFFFFFFFF]
    bits = np.zeros((5, E.WIDTH), dtype=np.uint32)
    bits[:, E.ENV] = envs
    bits[:, E.STEP] = [x & 0xFFFFFFFF for x in steps]
    bits[:, E.STEP + 1] = [x >> 32 for x in steps]
    d = decode_episode_records(torch.from_numpy(bits.view(np.float32)))
    want = sorted(zip(steps, envs))
    assert d["step"].tolist() == [w[0] for w in want] and d["env"].tolist() == [w[1] for w in want]


def _landing_targets(ora, n):
    """Half of the envs chase a target that sits where the drone was one step ago (so they land), half a fixed plate."""
    fixed = torch.tensor([0.5, -0.5, 0.377]).repeat(n, 1)
    chase = torch.arange(n) % 2 == 0
    return torch.where(chase[:, None], ora.root[:, 0:3].to(torch.float32), fixed)


@pytest.mark.parametrize("family", ["mode1", "mode2", "landing"])
def test_reference_tallies_equal_the_metrics(family):
    """300 steps at maxEpisodeLength 32: the records' count, lengths, time-outs, crash causes and landings are exactly the metrics
    reference's slots 9, 10, 11, 12, 13 and 2, and the exact sum of their returns is slot 1."""
    n, steps = 256, 300
    kw = dict(seed=3, max_episode_length=32, dr_enable=1, env_id_base=100)
    if family == "mode1":
        ora = E.with_episode_log(with_metrics(QuadStepOracle))(default_cfg(n, fault_mode=1, **kw))
    elif family == "mode2":
        cfg = default_cfg(n, fault_mode=2, fault_rotors_lo=0, fault_rotors_hi=4, fault_eff_lo=0.1, fault_eff_range=0.6,
                          fault_ramp_steps=5, **kw)
        ora = E.with_episode_log(with_metrics(M.MultiFaultOracle))(cfg)
    else:
        cfg = default_cfg(n, fault_mode=1, target_fixed=1, land_cutoff=0.2, plate_enable=1, plate_z=0.377, plate_radius=0.35,
                          die_z=0.3, **kw)
        ora = E.with_episode_log(with_metrics(QuadStepOracle))(cfg)
    g = torch.Generator().manual_seed(5)
    for t in range(steps):
        a = torch.rand(n, 4, generator=g) * 2 - 1
        if family == "landing":
            ora.step(a, target_in=_landing_targets(ora, n))
        else:
            ora.step(a)
    rows = ora.log_rows()
    tal = E.tallies(rows, last_step=steps - 1)
    for slot in (9, 10, 11, 12, 13, 2):
        assert tal[slot] == ora.counts[slot], (family, slot, tal[slot], ora.counts[slot])
    assert math.fsum(tal["returns"].tolist()) == ora.vector()[1]
    assert tal[9] > n and tal[11] > 0
    assert tal[2] > 0 if family == "landing" else tal[12] + tal[13] > 0
    if family == "mode2":
        eff = rows[:, E.EFF:E.EFF + 4].view(np.float32)
        assert ((eff != 1.0).sum(1) == 4).any() and ((eff == 1.0).all(1) == (rows[:, E.ONSET].view(np.int32) == -1)).all()
    assert (rows[:, E.RESERVED:] == 0).all()


def test_log_twins_meet_their_occupancy(lib):
    """generic log twins 6 CTAs/SM (at 7 they spill), sub-wave twins 4, TMA twins 5 with the states tile, at 128 threads; no spills
    (ptxas), no local memory, 228 KB of shared memory per SM with 1 KB per CTA reserved."""
    want = {"20quad_step_log_kernel": 6, "23quad_step_log_mf_kernel": 6, "28quad_step_log_subwave_kernel": 4,
            "31quad_step_log_mf_subwave_kernel": 4, "24quad_step_tma_log_kernel": 5, "27quad_step_tma_log_mf_kernel": 5}
    pat = r"_ZN3ozl(" + "|".join(want) + r")I(\w*?)EEv"
    seen = {}
    for name, r in _res_usage(lib).items():
        m = re.match(pat, name)
        if m:
            ctas = want[m.group(1)]
            seen.setdefault(m.group(1), []).append(m.group(2))
            assert r["LOCAL"] == 0, (name, r)
            assert r["REG"] * 128 * ctas <= 65536 and (r["SHARED"] + 1024) * ctas <= 228 * 1024, (name, r)
    # NONE / VEHICLE / LEE x states (mode 2: NONE / VEHICLE x states), TMA: x states
    assert {k: len(v) for k, v in seen.items()} == {"20quad_step_log_kernel": 6, "28quad_step_log_subwave_kernel": 6,
                                                    "23quad_step_log_mf_kernel": 4, "31quad_step_log_mf_subwave_kernel": 4,
                                                    "24quad_step_tma_log_kernel": 2, "27quad_step_tma_log_mf_kernel": 2}, seen
    spills = {k: v for k, v in _ptxas_spills().items() if re.match(pat, k)}
    assert len(spills) == 24 and all(v == (0, 0) for v in spills.values()), spills
