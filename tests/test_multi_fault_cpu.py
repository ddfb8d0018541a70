"""rotorFault mode "multi" (cfg.fault_mode 2), without a GPU: the header and binding layout, the config translation and its
refusals, the reset law on the CPU reference (tests/multi_fault_ref.py), known answers for the ramp, and the resources of the
fault_mode 2 kernel twins."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import multi_fault_ref as M
from oracle import philox as px
from oracle.quad_step import default_cfg


@pytest.fixture(scope="module")
def lib():
    from ouzelum_b200 import _lib
    return _lib


def test_header_and_binding_layout(lib):
    import ctypes as C
    L = lib.SCENARIO_LAYOUT
    assert lib.OZL_ABI_VERSION == 7 and lib.lib.ozl_abi_version() == 7
    assert lib.lib.ozl_cfg_size() == C.sizeof(lib.OzlCfg) == 408          # the ABI 6 size: the new fields use the reserved words
    assert (L["OZL_SCN_RFAULT_ONSET"], L["OZL_SCN_RFAULT_EFF"]) == (M.RONSET, M.REFF) == (26, 27)
    with open(os.path.join(os.path.dirname(lib.__file__), "csrc", "philox.cuh")) as f:
        assert re.search(r"P_RFAULT = (\d+)", f.read()).group(1) == str(M.P_RFAULT)
    c = lib.default_cfg(8)
    assert (c.fault_rotors_lo, c.fault_rotors_hi, c.fault_ramp_steps) == (1, 1, 0)


def _cfg(**fault):
    from ouzelum_b200.cfg import task_config
    from ouzelum_b200.tasks.ouzelum import x500_cfg_from_task
    return x500_cfg_from_task(task_config("Ouzelum", 16, rotorFault=dict({"enable": True}, **fault)), 16)


def test_config_translation_and_refusals(lib):
    c = _cfg()
    assert (c.fault_mode, c.fault_rotors_lo, c.fault_rotors_hi, c.fault_ramp_steps) == (1, 1, 1, 0)
    c = _cfg(mode="multi", rotors=[1, 3], effLow=0.2, effHigh=0.7, rampSteps=50)
    assert (c.fault_mode, c.fault_rotors_lo, c.fault_rotors_hi, c.fault_ramp_steps) == (2, 1, 3, 50)
    assert c.fault_eff_lo == pytest.approx(0.2) and c.fault_eff_range == pytest.approx(0.5)
    from ouzelum_b200.cfg import task_config
    from ouzelum_b200.tasks.ouzelum import x500_cfg_from_task
    assert x500_cfg_from_task(task_config("Ouzelum", 4, rotorFault={"mode": "multi"}), 4).fault_mode == 0     # not enabled
    for bad, text in [(dict(mode="double"), "mode"), (dict(mode="multi", rotors=[2, 1]), "rotors"),
                      (dict(mode="multi", rotors=[0, 5]), "rotors"), (dict(mode="multi", rotors=[-1, 2]), "rotors"),
                      (dict(mode="multi", rotors=[1]), "rotors"), (dict(mode="multi", rotors=[1.5, 2]), "rotors"),
                      (dict(mode="multi", rampSteps=-1), "rampSteps"), (dict(mode="multi", rampSteps=1 << 24), "rampSteps"),
                      (dict(mode="multi", effLow=0.5, effHigh=1.5), "effLow"), (dict(mode="multi", effLow=-0.1), "effLow")]:
        with pytest.raises(ValueError, match=text):
            _cfg(**bad)


def test_wrench_and_quadcopter_tasks_refuse_multi():
    from ouzelum_b200.tasks.ouzelum import refuse_multi_fault
    for name in ("LeeLanded", "EKFLeeLanded", "Quadcopter"):
        with pytest.raises(ValueError, match="multi"):
            refuse_multi_fault(name, {"rotorFault": {"enable": True, "mode": "multi"}})
        refuse_multi_fault(name, {"rotorFault": {"enable": True}})
    from ouzelum_b200.tasks import ekf_lee_landed, lee_landed, quadcopter
    import inspect
    for mod in (ekf_lee_landed, lee_landed, quadcopter):
        assert "refuse_multi_fault(" in inspect.getsource(mod)


def _mf_cfg(n, **kw):
    return default_cfg(n, **dict(dict(seed=5, fault_mode=2, fault_rotors_lo=0, fault_rotors_hi=4, fault_eff_lo=0.1,
                                      fault_eff_range=0.6, max_episode_length=300, env_id_base=1000), **kw))


def test_reset_law_on_the_reference():
    n = 24000
    cfg = _mf_cfg(n)
    ids = np.arange(n, dtype=np.uint64) + np.uint64(cfg["env_id_base"])
    onset, e, k, perm = M.reset_draw(cfg, ids, 17)
    assert int(k.min()) == 0 and int(k.max()) == 4
    assert sorted(set(perm.tolist())) == list(range(24))                # every permutation is reachable
    faulted = e != 1.0
    assert torch.equal(faulted.sum(1), k)                                # e < effHigh <= 1 for a faulted rotor here
    for kk in range(5):                                                  # the faulted set is the first k entries of the permutation
        i = int((k == kk).nonzero()[0])
        assert set(torch.nonzero(faulted[i]).flatten().tolist()) == set(M.PERMS[int(perm[i])][:kk])
    ev = e[faulted]
    assert float(ev.min()) >= np.float32(0.1) and float(ev.max()) < np.float32(0.7)
    assert torch.equal(onset[k == 0], torch.full_like(onset[k == 0], M.FAULT_NEVER))
    # the onset of a faulted episode is mode 1's onset for the same (seed, env, step)
    r1 = px.draw(cfg["seed"], ids, 17, px.P_FAULT)[1]
    m1 = torch.from_numpy(px.mulhi(r1, cfg["max_episode_length"]))
    assert torch.equal(onset[k > 0], m1[k > 0])
    # per-rotor fault frequencies and k are uniform (loose chi-square: 3 and 4 degrees of freedom, p ~ 1e-6)
    for counts, dof in ((faulted.sum(0).double(), 3), (torch.bincount(k, minlength=5).double(), 4)):
        exp = counts.sum() / len(counts)
        assert float(((counts - exp) ** 2 / exp).sum()) < 35.0, (counts, dof)
    # [lo, hi] = [2, 2]: exactly two rotors, never 'no fault'
    _, e2, k2, _ = M.reset_draw(_mf_cfg(512, fault_rotors_lo=2, fault_rotors_hi=2), ids[:512], 3)
    assert (k2 == 2).all() and ((e2 != 1.0).sum(1) == 2).all()


def test_ramp_known_answers():
    e = np.float32(0.25)
    for ramp in (0, 1):                                                  # abrupt
        for d in (0, 1, 7):
            assert M.ramp_factor(e, d, ramp) == e
    # ramp 4: x = (d + 1) * 0.25 exactly, a = fmaf(x, e - 1, 1) = 1 - 0.75 x
    assert [M.ramp_factor(e, d, 4) for d in range(5)] == [np.float32(0.8125), np.float32(0.625), np.float32(0.4375), e, e]
    # the vectorised form used by the oracle equals the scalar statement
    eff = torch.tensor([[0.25, 1.0, 0.6, 0.0]], dtype=torch.float32).repeat(9, 1)
    prog = torch.arange(9, dtype=torch.int64) + 3
    onset = torch.full((9,), 5, dtype=torch.int64)
    for ramp in (0, 1, 3, 7):
        a, active = M.factors(eff, onset, prog, ramp)
        for i in range(9):
            for j in range(4):
                want = M.ramp_factor(eff[i, j].item(), int(prog[i] - 5), ramp) if active[i] else np.float32(1.0)
                assert a[i, j].item() == want, (ramp, i, j)
        assert torch.equal(active, prog >= 5)
    # ramp 3, inv_ramp = (float)(1/3) rounded once: a differs from the exact 1 - (d+1)/3 (1 - e) by rounding only
    assert M.ramp_factor(np.float32(0.0), 0, 3) == np.float32(1.0) - np.float32(1.0 / 3.0)


def _res_usage(lib):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    out = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-res-usage", lib.LIB_PATH],
                         capture_output=True, text=True).stdout
    return {m.group(1): dict((k, int(v)) for k, v in re.findall(r"(\w+):(\d+)", m.group(2)))
            for m in re.finditer(r"Function (\S+):\s*\n\s*(REG:.*)", out)}


def _ptxas_spills():
    """{kernel: (spill store bytes, spill load bytes)} from a `-Xptxas -v` compile of quad_step.cu with the build's flags (on sm_100a
    a spill goes to the ABI stack frame, so cuobjdump's LOCAL column does not show it; ptxas does)."""
    import tempfile
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ozl_build_flags", os.path.join(here, "ouzelum_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([b.NVCC] + b.FLAGS + ["-Xptxas", "-v", "-c", "-o", os.path.join(d, "q.o"),
                                                 os.path.join(here, "ouzelum_b200", "csrc", "quad_step.cu")],
                           capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    out, cur = {}, None
    for line in (r.stdout + r.stderr).splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            out[cur] = (int(m.group(1)), int(m.group(2)))
            cur = None
    return out


def test_fault_mode_2_twins_meet_their_occupancy(lib):
    """generic twin 6 CTAs/SM (mode-2 launches switch to the TMA twin above one wave of it), sub-wave twin 4, TMA twin 5 (with the
    states tile) at 128 threads, no spills (ptxas) and no local memory; 228 KB of shared memory per SM including the 1 KB the driver
    reserves per CTA."""
    want = {"19quad_step_mf_kernel": 6, "27quad_step_mf_subwave_kernel": 4, "23quad_step_tma_mf_kernel": 5}
    pat = r"_ZN3ozl(19quad_step_mf_kernel|27quad_step_mf_subwave_kernel|23quad_step_tma_mf_kernel)I(\w*?)EEv"
    seen = {}
    for name, r in _res_usage(lib).items():
        m = re.match(pat, name)
        if m:
            ctas = want[m.group(1)]
            seen.setdefault(m.group(1), []).append(m.group(2))
            assert r["LOCAL"] == 0, (name, r)
            assert r["REG"] * 128 * ctas <= 65536 and (r["SHARED"] + 1024) * ctas <= 228 * 1024, (name, r)
    # FRONT_NONE and FRONT_VEHICLE, with and without the states output (TMA: FRONT_NONE only)
    assert {k: len(v) for k, v in seen.items()} == {"19quad_step_mf_kernel": 4, "27quad_step_mf_subwave_kernel": 4,
                                                    "23quad_step_tma_mf_kernel": 2}, seen
    spills = {k: v for k, v in _ptxas_spills().items() if re.match(pat, k) or "apply_resets_mf" in k}
    assert len(spills) == 11 and all(v == (0, 0) for v in spills.values()), spills
