"""Privileged critic state (ozl_set_states_output), without a GPU: the layout the header states, the CPU reference on hand-built
states with known answers, and the kernel instantiations the library carries."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import states_ref as R


@pytest.fixture(scope="module")
def lib():
    from ouzelum_b200 import _lib           # built by the session's native_library fixture
    return _lib


def test_header_layout_equals_the_reference_layout(lib):
    L = lib.STATES_LAYOUT
    assert lib.STATES_WIDTH == R.WIDTH == 32
    assert (L["OZL_STATE_OBS"], L["OZL_STATE_THRUST"], L["OZL_STATE_EFF"], L["OZL_STATE_MASS"], L["OZL_STATE_THRUST_SCALE"],
            L["OZL_STATE_YAW_KM"], L["OZL_STATE_PROGRESS"], L["OZL_STATE_POS"]) == \
        (R.OBS, R.THRUST, R.EFF, R.MASS, R.THRUST_SCALE, R.YAW_KM, R.PROGRESS, R.POS)
    assert (L["OZL_STATE_IXX"], L["OZL_STATE_IYY"], L["OZL_STATE_IZZ"], L["OZL_STATE_ARM"]) == (22, 23, 24, 25)


def test_states_row_known_answers():
    from oracle.quad_step import default_cfg
    cfg = default_cfg(3, max_episode_length=2000, clip_obs=5.0)
    f = lambda *v: torch.tensor(v, dtype=torch.float32)
    clean = torch.arange(39, dtype=torch.float32).reshape(3, 13) / 10.0 - 1.0
    root = torch.zeros(3, 13)
    root[:, 0:3] = f([3.0, -6.0, 30.0], [0.0, 0.0, 0.3], [1.5, 1.5, 1.5])
    thrust = f([0, 500, 1000, 2000], [0, 0, 0, 0], [2000, 2000, 2000, 2000])
    nominal = [float(np.float32(cfg[k])) for k in ("mass", "ixx", "iyy", "izz", "arm")]
    params7 = torch.tensor([nominal + [1.0, 0.0], [2 * v for v in nominal] + [1.1, 0.016], nominal + [0.9, 7.0]], dtype=torch.float32)
    active = torch.tensor([False, True, True])
    rotor, eff = torch.tensor([2, 2, 0]), f(0.3, 0.3, 0.25)
    prog = torch.tensor([500, 1, 2000])
    s = R.states_row(clean, root, thrust, active, rotor, eff, params7, prog, cfg)
    assert s.shape == (3, 32) and s.dtype == torch.float32
    assert torch.equal(s[:, 0:13], torch.clamp(clean, -5, 5))
    assert s[0, 13:17].tolist() == [0.0, 0.25, 0.5, 1.0] and s[2, 13:17].tolist() == [1.0] * 4
    assert s[0, 17:21].tolist() == [1.0] * 4                        # fault not active: all ones
    assert s[1, 17:21].tolist() == [1.0, 1.0, np.float32(0.3), 1.0]
    assert s[2, 17:21].tolist() == [np.float32(0.25), 1.0, 1.0, 1.0]
    assert s[0, 21:27].tolist() == [1.0] * 6                         # nominal parameters: exactly 1
    assert s[1, 21:26].tolist() == [2.0] * 5 and s[1, 26].item() == np.float32(1.1)
    assert s[1, 27].item() == np.float32(0.016) and s[2, 27].item() == 5.0      # yaw_km raw, clamped
    assert s[0, 28].item() == 0.25 and s[2, 28].item() == 1.0 and s[1, 28].item() == np.float32(1) / np.float32(2000)
    inv3 = np.float32(1) / np.float32(3)
    assert s[0, 29:32].tolist() == [np.float32(3) * inv3, np.float32(-6) * inv3, 5.0]       # /3 scaling, then the clamp
    assert s[1, 31].item() == np.float32(0.3) * inv3


def test_oracle_states_carry_the_clean_observation():
    """With no sensor-fault model the clean observation IS the delivered one; with it, the two differ while the states do not."""
    from oracle.quad_step import default_cfg
    g = torch.Generator().manual_seed(3)
    rows = {}
    for mode in (0, 3):
        ora = R.StatesOracle(default_cfg(64, seed=11, fault_mode=1, dr_enable=1, pomdp_mode=mode, pomdp_prob=0.3, noise_sigma=0.2,
                                         max_episode_length=12))
        g.manual_seed(3)
        for _ in range(15):
            ora.step((torch.rand(64, 4, generator=g) * 2 - 1) * 0.3)
            if mode == 0:
                assert torch.equal(ora.states_buf[:, 0:13], ora.obs_buf)
        rows[mode] = (ora.states_buf.clone(), ora.obs_buf.clone())
    assert torch.equal(rows[0][0], rows[3][0])
    assert not torch.equal(rows[3][0][:, 0:13], rows[3][1])


def _res_usage(lib):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    out = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-res-usage", lib.LIB_PATH],
                         capture_output=True, text=True).stdout
    return {m.group(1): dict((k, int(v)) for k, v in re.findall(r"(\w+):(\d+)", m.group(2)))
            for m in re.finditer(r"Function (\S+):\s*\n\s*(REG:.*)", out)}


def test_library_carries_both_step_instantiations_without_extra_local_memory(lib):
    """Both instantiations of every step kernel exist; the states output adds no stack / local memory, keeps the register budget
    of the occupancy target (generic 7 x 128-thread CTAs / SM, TMA kernel 5) and its shared memory fits that many CTAs per SM
    (228 KB of shared memory per B200 SM; the figures include the 1 KB the driver reserves per CTA)."""
    ru = _res_usage(lib)
    pairs = {}
    for name, r in ru.items():
        m = re.match(r"_ZN3ozl(?:16quad_step_kernelILi128ELi(\d)E|20quad_step_tma_kernelI)Lb([01])E", name)
        if m:
            pairs.setdefault(m.group(1) or "tma", {})[m.group(2)] = r
    assert sorted(pairs) == ["0", "1", "2", "tma"], sorted(pairs)
    for kind, p in pairs.items():
        off, on = p["0"], p["1"]
        ctas = 5 if kind == "tma" else 7
        assert on["STACK"] == off["STACK"] and on["LOCAL"] == off["LOCAL"] == 0, (kind, off, on)
        assert on["REG"] * 128 * ctas <= 65536, (kind, on)
        assert on["SHARED"] * ctas <= 228 * 1024, (kind, on)
        assert on["SHARED"] >= off["SHARED"] + 128 * 32 * 4, (kind, off, on)        # the 16 KB states tile


def test_set_states_output_needs_a_handle(lib):
    L = lib.lib
    assert L.ozl_set_states_output(None, None, 32) != 0 and "env is NULL" in L.ozl_last_error().decode()
