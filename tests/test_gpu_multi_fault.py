"""rotorFault mode "multi" (cfg.fault_mode 2) on the GPU: the fault_mode 2 kernel twins (generic, sub-wave, TMA + ragged tail) equal
the CPU reference (tests/multi_fault_ref.py) bit for bit over many resets, ramp or not, with the states row, scenario tables and the
metrics vector; mode 2 pinned to one rotor reproduces mode 1 exactly; the other step paths, ozl_apply_resets, sharding, CUDA-graph
replay and checkpoints follow the law; every refusal holds."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import multi_fault_ref as M
import scenario_ref as S
from metrics_ref import assert_metrics, with_metrics

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MF = dict(seed=7, fault_mode=2, fault_rotors_lo=0, fault_rotors_hi=3, fault_eff_lo=0.05, fault_eff_range=0.6, dr_enable=1,
          max_episode_length=32, target_period=9, lin_drag=0.05, yaw_km=0.016, env_id_base=321)


class _kernel_env:
    """OZL_TMA_MIN_TILES / OZL_EARLY_DRAW_MAX_ENVS (read at ozl_create) for the handles created inside: tma True forces the TMA twin
    (False never), early False keeps launches off the sub-wave twin (so 4099 envs run the generic twin over a full grid)."""

    def __init__(self, tma=None, early=None):
        self.set = {}
        if tma is not None:
            self.set["OZL_TMA_MIN_TILES"] = "1" if tma else "0"
        if early is not None and not early:
            self.set["OZL_EARLY_DRAW_MAX_ENVS"] = "0"

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.set}
        os.environ.update(self.set)

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _mk(n, tma=None, rows=None, states=True, early=None, **kw):
    from ouzelum_b200 import _lib
    from ouzelum_b200.sim import QuadSim
    with _kernel_env(tma, early):
        cfg = _lib.default_cfg(n, **kw)
        sim = QuadSim(cfg, DEV)
    b = dict(obs=torch.zeros(n, 13, device=DEV), rew=torch.zeros(n, device=DEV),
             reset=torch.ones(n, dtype=torch.int64, device=DEV), progress=torch.zeros(n, dtype=torch.int64, device=DEV),
             timeout=torch.zeros(n, dtype=torch.uint8, device=DEV), ep_ret=torch.zeros(n, device=DEV))
    if states:
        b["states"] = torch.full((n, 32), float("nan"), device=DEV)
        sim.set_states_output(b["states"])
    if rows is not None:
        sim.set_scenarios(rows)
    return sim, b, cfg


def _step(sim, b, a):
    sim.step(a, b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])


def _actions(n, t, scale=0.3):
    g = torch.Generator().manual_seed(2000 + t)
    return ((torch.rand(n, 4, generator=g) * 2 - 1) * scale).to(DEV)


def mf_rows(n, seed=0):
    """Every 3rd env pinned to a multi-rotor fault (some 'no fault': four 1s), every 3rd + 1 also partly pinned elsewhere."""
    g = torch.Generator().manual_seed(seed)
    rows = S.empty(n)
    full, part = torch.arange(n) % 3 == 0, torch.arange(n) % 3 == 1
    e = torch.rand(n, 4, generator=g)
    e = torch.where(torch.rand(n, 4, generator=g) < 0.5, e, torch.ones(()))
    rows[full, M.RONSET] = torch.randint(0, 20, (n,), generator=g).float()[full]
    rows[full, M.REFF:M.REFF + 4] = e[full]
    rows[part, 0:3] = torch.tensor([0.3, -0.2, 1.5])
    rows[part, S.MASS] = 2.3
    return rows


def _oracle(cfg, rows=None):
    return with_metrics(M.MultiFaultOracle)(cfg.to_dict(), rows)


def _compare(sim, b, ora, t, full=False):
    for k, o in (("obs", ora.obs_buf), ("rew", ora.rew_buf), ("reset", ora.reset_buf), ("progress", ora.progress_buf),
                 ("timeout", ora.timeout_buf.to(torch.uint8)), ("states", ora.states_buf if "states" in b else None)):
        if o is not None:
            assert torch.equal(b[k].cpu(), o), f"t={t}: {k}"
    if full:
        st = sim.get_state()
        assert torch.equal(st["root"].cpu(), ora.root) and torch.equal(st["thrust"].cpu(), ora.thrust), t
        eff = sim.get_rotor_eff().cpu()
        assert torch.equal(eff, ora.rotor_eff), t
        assert torch.equal((sim.get_params()[1].cpu()[:, 1].long() & M.FAULT_NEVER), ora.fault_onset), t


@pytest.mark.parametrize("n,tma,early,ramp,table,states", [
    (4099, False, False, 0, False, False), (4099, False, False, 9, True, True),        # generic twin over the whole grid
    (4099, False, None, 0, True, False), (16384, None, None, 9, False, True),          # sub-wave twin
    (132608 + 77, True, None, 9, True, True)])                                          # TMA twin + ragged tail (generic twin)
def test_kernels_equal_the_reference(n, tma, early, ramp, table, states):
    """generic (4099 with the sub-wave twin off), sub-wave (4099, 16384: one wave of 4 CTAs per SM) and TMA + ragged tail (132685),
    with and without a table and the states output: 200 steps, maxEpisodeLength 32."""
    from ouzelum_b200 import _lib
    kw = dict(MF, fault_ramp_steps=ramp, dr={5: (_lib.DR_GAUSSIAN, _lib.DR_SCALING, 1.0, 0.05)})
    rows = mf_rows(n, seed=n) if table else None
    sim, b, cfg = _mk(n, tma=tma, rows=rows, states=states, early=early, **kw)
    ora = _oracle(cfg, rows)
    ramping = faulted = 0
    for t in range(200):
        a = _actions(n, t)
        _step(sim, b, a)
        ora.step(a.cpu())
        _compare(sim, b, ora, t, full=(t % 50 == 49))
        s = ora.applied_eff
        if states:
            assert torch.equal(b["states"].cpu()[:, 17:21], s), t
        faulted += int((s != 1.0).any(1).sum())
        ramping += int(((s != 1.0) & (s != ora.rotor_eff)).any(1).sum())
    assert_metrics(sim.metrics(), ora, f"n={n}")
    assert faulted > 0 and int(ora.counts[14]) > 0 and int(ora.counts[9]) > n
    assert (ramping > 0) == (ramp > 1)


def test_mode_2_pinned_to_one_rotor_is_mode_1():
    """A mode-1 row (rotor r, onset o, eff e) and the mode-2 row (onset o, e at r, 1 elsewhere), ramp 0: the same results."""
    n = 4099
    g = torch.Generator().manual_seed(3)
    rotor = torch.randint(-1, 4, (n,), generator=g)
    onset = torch.randint(0, 25, (n,), generator=g).float()
    eff = torch.rand(n, generator=g) * 0.9
    r1, r2 = S.empty(n), S.empty(n)
    r1[:, 16], r1[:, 17], r1[:, 18] = rotor.float(), onset, eff
    e4 = torch.ones(n, 4)
    hit = rotor >= 0
    e4[hit.nonzero()[:, 0], rotor[hit]] = eff[hit]
    r2[:, M.RONSET], r2[:, M.REFF:M.REFF + 4] = onset, e4
    kw = {k: v for k, v in MF.items() if not k.startswith("fault_rotors")}
    s1, b1, _ = _mk(n, rows=r1, **dict(kw, fault_mode=1))
    s2, b2, _ = _mk(n, rows=r2, **dict(kw, fault_mode=2))
    for t in range(150):
        a = _actions(n, t)
        _step(s1, b1, a)
        _step(s2, b2, a)
        for k in b1:
            assert torch.equal(b1[k], b2[k]), (t, k)
    assert torch.equal(s1.metrics(), s2.metrics())
    assert torch.equal(s1.get_state()["root"], s2.get_state()["root"])
    assert int(s1.metrics()[14].item()) > 0


def test_other_step_paths_and_apply_resets():
    """ozl_step_tracking, ozl_step_host_sync and ozl_step_wrench against the reference; ozl_apply_resets writes the draw of the
    next step; ozl_landing_step reports a_j of its own state by the law."""
    from ouzelum_b200._lib import OzlHostIo, lib
    n = 1000
    sim, b, cfg = _mk(n, early=False, **dict(MF, fault_ramp_steps=4))       # the generic twin (dispatch of launch_step_t)
    ora = _oracle(cfg)
    pin = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt).pin_memory()
    ah, oh, rh, dh, xh = pin(n, 4), pin(n, 13), pin(n), pin(n, dt=torch.uint8), pin(n, dt=torch.int64)
    io = OzlHostIo(ah.data_ptr(), oh.data_ptr(), rh.data_ptr(), dh.data_ptr(), xh.data_ptr(), b["reset"].data_ptr(),
                   b["progress"].data_ptr(), b["timeout"].data_ptr(), b["ep_ret"].data_ptr())
    tgt = torch.tensor([0.5, -0.5, 1.2]).repeat(n, 1)
    for t in range(90):
        a = _actions(n, t)
        path = t % 3
        if path == 0:
            sim.step_tracking(a, tgt.to(DEV), b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])
            ora.step(a.cpu(), target_in=tgt)
        elif path == 1:
            ah.copy_(a.cpu())
            assert lib.ozl_step_host_sync(sim._h, C.byref(io), torch.cuda.current_stream().cuda_stream) == 0
            b["obs"].copy_(oh)
            b["rew"].copy_(rh)
            ora.step(a.cpu())
        else:
            w = torch.cat([a[:, :1] * 20 + 20, a[:, 1:] * 0.01], 1).contiguous()
            sim.step_wrench(w, None, b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])
            ora.step(w.cpu(), act_mode=1)
        _compare(sim, b, ora, t, full=(t % 10 == 9))
        if t % 10 == 5:
            sim.apply_resets(b["reset"])
            r = (b["reset"] != 0).cpu()
            onset, e = ora.pending_reset()
            assert torch.equal(sim.get_rotor_eff().cpu()[r], e[r]), t
            assert torch.equal(sim.get_params()[1].cpu()[r, 1].long() & M.FAULT_NEVER, onset[r]), t
    assert_metrics(sim.metrics(), ora, "paths")
    # ozl_landing_step (FRONT_VEHICLE twins, generic and sub-wave) against the reference fed the vehicle's target
    for early in (False, None):
        with _kernel_env(early=early):
            env = _task("Landing", 1500, rotorFault={"enable": True, "mode": "multi", "rotors": [1, 4], "rampSteps": 6},
                        domainRandomization={"enable": True}, asymmetric_observations=True)
        lo = with_metrics(M.MultiFaultOracle)(env.native_cfg.to_dict())
        seen = 0
        for t in range(80):
            a = _actions(1500, t)
            env.step(a)
            lo.step(a.cpu(), target_in=env.husky.target.cpu())
            for k, got, want in (("obs", env.obs_buf, lo.obs_buf), ("rew", env.rew_buf, lo.rew_buf),
                                 ("reset", env.reset_buf, lo.reset_buf), ("progress", env.progress_buf, lo.progress_buf),
                                 ("states", env.states_buf, lo.states_buf)):
                assert torch.equal(got.cpu(), want), (early, t, k)
            seen += int((lo.applied_eff != 1).any(1).sum())
        assert torch.equal(env.sim.get_rotor_eff().cpu(), lo.rotor_eff)
        assert torch.equal(env.sim.get_state()["root"].cpu(), lo.root)
        assert_metrics(env.metrics(), lo, f"Landing early={early}")
        assert seen > 0


def test_shards_and_graph_replay():
    n, h = 4096, 2048
    rows = mf_rows(n, seed=9)
    kw = dict(MF, fault_ramp_steps=7)
    full, bf, _ = _mk(n, rows=rows, **dict(kw, env_id_base=0))
    lo, bl, _ = _mk(h, rows=rows[:h].clone(), **dict(kw, env_id_base=0))
    hi, bh, _ = _mk(h, rows=rows[h:].clone(), **dict(kw, env_id_base=h))
    gr, bg, _ = _mk(n, rows=rows, **dict(kw, env_id_base=0))
    static_a = torch.zeros(n, 4, device=DEV)
    _step(gr, bg, static_a)                                  # warm-up launch outside the capture; the eager handle takes it too
    _step(full, bf, static_a)
    _step(lo, bl, static_a[:h].contiguous())
    _step(hi, bh, static_a[h:].contiguous())
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _step(gr, bg, static_a)
    for t in range(100):
        a = _actions(n, t)
        _step(full, bf, a)
        _step(lo, bl, a[:h].contiguous())
        _step(hi, bh, a[h:].contiguous())
        static_a.copy_(a)
        g.replay()
        for k in ("obs", "rew", "reset", "states"):
            assert torch.equal(bf[k], torch.cat([bl[k], bh[k]])), (t, k)
            assert torch.equal(bf[k], bg[k]), (t, k)
    assert torch.equal(full.get_rotor_eff(), torch.cat([lo.get_rotor_eff(), hi.get_rotor_eff()]))
    assert torch.equal(full.get_rotor_eff(), gr.get_rotor_eff())


def _task(name, n, **env):
    import ouzelum_b200
    cfg = ouzelum_b200.task_config(name, n, seed=5, maxEpisodeLength=30, **env)
    return ouzelum_b200.make(seed=5, task=name, num_envs=n, sim_device=DEV, rl_device=DEV, headless=True, cfg=cfg)


def test_checkpoint_mid_ramp_continues_bit_identically():
    n = 500
    kw = dict(rotorFault={"enable": True, "mode": "multi", "rotors": [2, 4], "rampSteps": 25}, domainRandomization={"enable": True},
              asymmetric_observations=True)
    env = _task("Ouzelum", n, **kw)
    for t in range(23):
        env.step(_actions(n, t))
    sd = env.state_dict()
    assert sd["rotor_eff"].shape == (n, 4) and bool((sd["rotor_eff"] != 1).any())
    s = env.states_buf.cpu()[:, 17:21]
    assert bool(((s != 1) & (s != sd["rotor_eff"])).any())               # some env is inside its ramp
    env2 = _task("Ouzelum", n, **kw)
    env2.load_state_dict(sd)
    for t in range(23, 70):
        a = _actions(n, t)
        o1, r1, d1, _ = env.step(a)
        o2, r2, d2, _ = env2.step(a)
        assert torch.equal(o1["obs"], o2["obs"]) and torch.equal(o1["states"], o2["states"]), t
        assert torch.equal(r1, r2) and torch.equal(d1, d2), t
    single = _task("Ouzelum", n, rotorFault={"enable": True})
    with pytest.raises(ValueError, match="multi"):
        single.load_state_dict(sd)
    with pytest.raises(ValueError, match="multi"):
        env2.load_state_dict(single.state_dict())


def test_refusals_and_validation():
    from ouzelum_b200 import _lib
    from ouzelum_b200._lib import OzlEkfLeeArgs, OzlHuskyArgs, OzlLeeLandedArgs, lib
    from ouzelum_b200.sim import QuadSim
    n = 64
    msg = lambda: lib.ozl_last_error().decode()
    sim, b, _ = _mk(n, states=False, **MF)
    assert lib.ozl_rollout(sim._h, 4, b["obs"].data_ptr(), b["rew"].data_ptr(), b["reset"].data_ptr(), b["progress"].data_ptr(),
                           None) != 0 and "fault_mode 2" in msg()
    husky, gains = OzlHuskyArgs(), (C.c_float * 16)()
    args = OzlLeeLandedArgs(gains, (C.c_float * 4)(0, 0, 1, 0), 19.62, None)
    assert lib.ozl_lee_landed_step(sim._h, C.byref(args), C.byref(husky), b["obs"].data_ptr(), b["rew"].data_ptr(),
                                   b["reset"].data_ptr(), b["progress"].data_ptr(), None, None, None) != 0 and "fault_mode 2" in msg()
    assert lib.ozl_ekf_lee_landed_step(sim._h, C.byref(OzlEkfLeeArgs()), C.byref(husky), b["obs"].data_ptr(), b["rew"].data_ptr(),
                                       b["reset"].data_ptr(), b["progress"].data_ptr(), None, None, None) != 0 and "fault_mode 2" in msg()
    # the per-rotor effectiveness exists in mode 2 only
    single, _, _ = _mk(n, states=False, **dict(MF, fault_mode=1))
    for fn in (single.get_rotor_eff, lambda: single.set_rotor_eff(torch.ones(n, 4))):
        with pytest.raises(ValueError, match="fault_mode"):
            fn()
    sim.set_rotor_eff(torch.full((n, 4), 0.5))
    assert bool((sim.get_rotor_eff() == 0.5).all())
    # ozl_create
    for over, text in [(dict(fault_rotors_lo=3, fault_rotors_hi=2), "fault_rotors_lo"), (dict(fault_rotors_hi=5), "fault_rotors_lo"),
                       (dict(fault_ramp_steps=1 << 24), "fault_ramp_steps"), (dict(fault_ramp_steps=-2), "fault_ramp_steps"),
                       (dict(fault_eff_lo=-0.5), "fault_eff_lo -0.5 is not in"), (dict(fault_eff_lo=0.5, fault_eff_range=0.6), "fault_eff_range")]:
        with pytest.raises(RuntimeError, match=text):
            QuadSim(_lib.default_cfg(n, **dict(MF, **over)), DEV)

    def bad(rows_edit, text, s=sim):
        r = S.empty(n)
        rows_edit(r)
        with pytest.raises(ValueError, match=text):
            s.set_scenarios(r)

    def put(first, vals):
        def f(r):
            r[3, first:first + len(vals)] = torch.tensor(vals, dtype=torch.float32)
        return f
    bad(put(16, [1.0, 0.0, 0.5]), "rotor faults group \\(slots 26-30\\)")
    bad(put(26, [2.0, 0.5, 1.0, 1.0, math.nan]), "rotor faults group must be all NaN or all set")
    bad(put(26, [2.0, 0.5, 1.0, 1.0, math.inf]), "rotor faults group has a non-finite")
    bad(put(26, [2.5, 0.5, 1.0, 1.0, 1.0]), "rotor faults onset")
    bad(put(26, [float(1 << 24), 0.5, 1.0, 1.0, 1.0]), "rotor faults onset")
    bad(put(26, [-1.0, 0.5, 1.0, 1.0, 1.0]), "rotor faults onset")
    bad(put(26, [2.0, 0.5, 1.0, 1.5, 1.0]), "effectiveness 1.5 of rotor 2")
    bad(put(26, [2.0, 0.5, -0.1, 1.0, 1.0]), "effectiveness -0.1 of rotor 1")
    bad(put(31, [0.0]), "reserved slot 31")
    bad(put(27, [0.5]), "reserved slot 27 .*fault_mode 2", s=single)
    sim.set_scenarios(mf_rows(n, seed=1))                   # a valid mode-2 table registers
    for name in ("LeeLanded", "EKFLeeLanded", "Quadcopter"):
        with pytest.raises(ValueError, match="multi"):
            _task(name, 64, rotorFault={"enable": True, "mode": "multi"})
    from ouzelum_b200 import scenarios
    rows = scenarios.multi_fault_grid(n, [(0.5, 1, 1, 1), (0.2, 0.3, 1, 0.9)], [0, 10])
    sim.set_scenarios(rows)
    assert rows[1, 26].item() == 10.0 and rows[2, 27:31].tolist() == pytest.approx([0.2, 0.3, 1, 0.9])
