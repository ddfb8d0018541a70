"""Episode log (ozl_set_episode_log) on the GPU: the log twins of the generic, sub-wave and TMA (+ ragged tail) step kernels write the
CPU reference's record set (tests/episode_log_ref.py) bit for bit, with faults off, mode 1 and mode 2 with a ramp, with and without a
scenario table and the states output; every other output equals a run without the log; the records tally with the same run's
metrics; the other step paths, sharding, CUDA-graph replay and overflow follow the law; every refusal holds."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import episode_log_ref as E
import multi_fault_ref as M
import scenario_ref as S
from metrics_ref import assert_metrics, with_metrics
from test_gpu_multi_fault import _kernel_env, mf_rows

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BASE = dict(seed=9, dr_enable=1, max_episode_length=32, target_period=9, lin_drag=0.05, yaw_km=0.016, env_id_base=555,
            fault_eff_lo=0.05, fault_eff_range=0.6)
FAULTS = {0: dict(fault_mode=0), 1: dict(fault_mode=1), 2: dict(fault_mode=2, fault_rotors_lo=0, fault_rotors_hi=3, fault_ramp_steps=9)}


def _mk(n, log, tma=None, early=None, rows=None, states=True, capacity=None, **kw):
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
    if log:
        sim.records = torch.zeros(capacity or 40 * n, 32, device=DEV)
        sim.head = torch.zeros(1, dtype=torch.int64, device=DEV)
        sim.set_episode_log(sim.records, sim.head)
    return sim, b, cfg


def _step(sim, b, a):
    sim.step(a, b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])


def _actions(n, t, scale=0.6):
    g = torch.Generator().manual_seed(3000 + t)
    return ((torch.rand(n, 4, generator=g) * 2 - 1) * scale).to(DEV)


def _read(sim, clear=False):
    """(uint32 [min(head, capacity), 32] sorted by (step, env), head)"""
    head = int(sim.head.item())
    k = min(head, sim.records.shape[0])
    bits = sim.records[:k].cpu().numpy().view(np.uint32)
    if clear:
        sim.head.zero_()
    return E.sort_rows(bits), head


def _same_rows(got, want, tag):
    assert got.shape == want.shape, f"{tag}: {got.shape[0]} records, reference {want.shape[0]}"
    bad = np.nonzero((got != want).any(1))[0]
    assert len(bad) == 0, f"{tag}: record {bad[0]} differs in slots {np.nonzero(got[bad[0]] != want[bad[0]])[0].tolist()}"


def _oracle(cfg, rows):
    d = cfg.to_dict()
    if d["fault_mode"] == 2:
        return E.with_episode_log(with_metrics(M.MultiFaultOracle))(d, rows)
    return E.with_episode_log(with_metrics(S.ScenarioOracle))(d, S.empty(d["num_envs"]) if rows is None else rows)


def _metric_tallies(sim, bits, last_step):
    m = sim.metrics().cpu().numpy()
    tal = E.tallies(bits, last_step=last_step)
    for slot in (9, 10, 11, 12, 13, 2):
        assert tal[slot] == m[slot], (slot, tal[slot], m[slot])
    ret = tal["returns"].tolist()           # slot 1 within metrics_ref's bound of a float64 sum in any order
    assert abs(m[1] - math.fsum(ret)) <= max(len(ret) - 1, 0) * 2.0 ** -53 * math.fsum(abs(x) for x in ret)


@pytest.mark.parametrize("n,tma,early,fault,table,states", [
    (37, None, None, 0, False, False),                     # sub-wave, one ragged warp
    (4099, False, False, 1, True, True),                   # generic twin over the whole grid
    (4099, False, False, 2, False, False),                 # generic mode-2 twin
    (16384, None, None, 2, True, True),                    # sub-wave mode-2 twin (the default at 16384)
    (16384, None, None, 1, False, True),                   # sub-wave twin
    (96037, True, None, 1, True, True),                    # TMA twin, several tiles per CTA, + ragged tail
    (96037, True, None, 2, False, True)])                  # TMA mode-2 twin + ragged tail
def test_log_equals_the_reference(n, tma, early, fault, table, states):
    """200 steps at maxEpisodeLength 32: the record set is the reference's bit for bit, and every other output -- obs, reward, reset,
    progress, time-outs, episode return, stored state, params, rotor effectiveness, states rows, metrics -- equals the same run
    without the log."""
    from ouzelum_b200 import _lib
    kw = dict(BASE, **FAULTS[fault])
    rows = (mf_rows(n, seed=n) if fault == 2 else S.mixed_rows(n, _lib.default_cfg(n, **kw).to_dict(), seed=n)) if table else None
    sim, b, cfg = _mk(n, True, tma=tma, early=early, rows=rows, states=states, **kw)
    ref, rb, _ = _mk(n, False, tma=tma, early=early, rows=rows, states=states, **kw)
    ora = _oracle(cfg, rows)
    for t in range(200):
        a = _actions(n, t)
        _step(sim, b, a)
        _step(ref, rb, a)
        ora.step(a.cpu())
        for k in b:
            assert torch.equal(b[k], rb[k]), (t, k)
    got, head = _read(sim)
    _same_rows(got, ora.log_rows(), f"n={n} fault={fault}")
    assert head == len(got) > n
    assert torch.equal(sim.metrics(), ref.metrics())
    assert_metrics(sim.metrics(), ora, f"n={n}")
    _metric_tallies(sim, got, 199)
    for x, y in ((sim.get_state()["root"], ref.get_state()["root"]), (sim.get_params()[0], ref.get_params()[0]),
                 (sim.get_params()[1], ref.get_params()[1])):
        assert torch.equal(x, y)
    if fault == 2:
        assert torch.equal(sim.get_rotor_eff(), ref.get_rotor_eff())
    flags = got[:, E.FLAGS]
    assert ((flags & E.TIMEOUT) != 0).any() and (n < 4096 or ((flags & (E.CRASH_DIST | E.CRASH_Z)) != 0).any())
    if fault:
        assert ((flags & E.FAULT_ACTIVE) != 0).any()


def _records_from_state(sim, b, step, mode, act_mode=0):
    """The records of the envs flagged for reset after a step, from the handle's own post-step state (get_state / get_params /
    get_rotor_eff) -- the reference for step paths whose front the CPU oracle does not model (the Lee controller)."""
    done = (b["reset"] != 0).cpu().numpy()
    n = done.shape[0]
    st = sim.get_state()
    p8, f2 = (x.cpu() for x in sim.get_params())
    root, tgt = st["root"].cpu(), st["target"].cpu()
    prog = b["progress"].cpu().numpy()
    onset = (f2[:, 1].numpy().astype(np.int64) & E.FAULT_NEVER)
    landed = f2[:, 1].numpy() < 0
    active = (prog - 1 >= onset) if (mode and act_mode == 0) else np.zeros(n, dtype=bool)
    if mode == 2:
        eff = sim.get_rotor_eff().cpu().numpy()
    else:
        eff = np.ones((n, 4), dtype=np.float32)
        if mode == 1:
            hit = onset != E.FAULT_NEVER
            eff[hit, f2[:, 0].numpy()[hit]] = p8[:, 6].numpy()[hit]
    dist = E.dist32(tgt, root[:, 0:3])
    cfg = sim.cfg
    flags = (b["timeout"].cpu().numpy().astype(np.uint32) * E.TIMEOUT | (dist > np.float32(cfg.die_dist)) * E.CRASH_DIST
             | (root[:, 2].numpy() < np.float32(cfg.die_z)) * E.CRASH_Z | landed * E.LANDED | active * E.FAULT_ACTIVE).astype(np.uint32)
    r = np.zeros((n, 32), dtype=np.uint32)
    r[:, E.ENV] = np.arange(n, dtype=np.uint32) + np.uint32(cfg.env_id_base)
    r[:, E.LENGTH] = prog.astype(np.uint32)
    r[:, E.STEP] = step
    r[:, E.RETURN] = E.f32_bits(b["ep_ret"].cpu().numpy())
    r[:, E.FLAGS] = flags
    r[:, E.ONSET] = np.where(onset == E.FAULT_NEVER, -1, onset).astype(np.uint32)
    r[:, E.DIST] = E.f32_bits(dist)
    r[:, E.EFF:E.EFF + 4] = E.f32_bits(eff)
    r[:, E.MASS:E.MASS + 7] = E.f32_bits(torch.cat([p8[:, 0:6], p8[:, 7:8]], 1).numpy())
    r[:, E.POS:E.POS + 3] = E.f32_bits(root[:, 0:3].numpy())
    r[:, E.LINVEL:E.LINVEL + 3] = E.f32_bits(root[:, 7:10].numpy())
    r[:, E.TARGET:E.TARGET + 3] = E.f32_bits(tgt.numpy())
    return r[done]


def test_other_step_paths():
    """ozl_step_tracking, ozl_step_host_sync, ozl_step_host_launch + ozl_step_host_wait (the completion word) and ozl_step_wrench
    (generic twin) against the reference; ozl_apply_resets writes no record."""
    from ouzelum_b200._lib import OzlHostIo, lib
    n = 1000
    for fault in (1, 2):
        sim, b, cfg = _mk(n, True, early=False, **dict(BASE, **FAULTS[fault]))
        ora = _oracle(cfg, None)
        pin = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt).pin_memory()
        ah, oh, rh, dh, xh = pin(n, 4), pin(n, 13), pin(n), pin(n, dt=torch.uint8), pin(n, dt=torch.int64)
        io = OzlHostIo(ah.data_ptr(), oh.data_ptr(), rh.data_ptr(), dh.data_ptr(), xh.data_ptr(), b["reset"].data_ptr(),
                       b["progress"].data_ptr(), b["timeout"].data_ptr(), b["ep_ret"].data_ptr())
        tgt = torch.tensor([0.5, -0.5, 1.2]).repeat(n, 1)
        for t in range(120):
            a = _actions(n, t)
            path = t % 3
            if path == 0:
                sim.step_tracking(a, tgt.to(DEV), b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])
                ora.step(a.cpu(), target_in=tgt)
            elif path == 1:
                ah.copy_(a.cpu())
                st = torch.cuda.current_stream().cuda_stream
                if (t // 3) % 2:
                    assert lib.ozl_step_host_launch(sim._h, C.byref(io), st) == 0 and lib.ozl_step_host_wait(sim._h, st) == 0
                else:
                    assert lib.ozl_step_host_sync(sim._h, C.byref(io), st) == 0
                ora.step(a.cpu())
            else:
                w = torch.cat([a[:, :1] * 20 + 20, a[:, 1:] * 0.01], 1).contiguous()
                sim.step_wrench(w, None, b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])
                ora.step(w.cpu(), act_mode=1)
            if t % 10 == 5:
                before = int(sim.head.item())
                sim.apply_resets(b["reset"])
                assert int(sim.head.item()) == before
        _same_rows(_read(sim)[0], ora.log_rows(), f"paths fault={fault}")


@pytest.mark.parametrize("fault", [1, 2])
def test_tma_many_tiles_per_cta(fault):
    """The TMA twins with three tiles per resident CTA and a ragged tail: each step's records are those of the handle's own post-step
    state, and every output equals a run without the log."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 3 * 5 * sms * 128 + 77
    kw = dict(BASE, **FAULTS[fault])
    sim, b, _ = _mk(n, True, tma=True, capacity=n * 8, **kw)
    ref, rb, _ = _mk(n, False, tma=True, **kw)
    want = []
    for t in range(60):
        a = _actions(n, t)
        _step(sim, b, a)
        _step(ref, rb, a)
        for k in b:
            assert torch.equal(b[k], rb[k]), (t, k)
        want.append(_records_from_state(sim, b, t, fault))
    got, head = _read(sim)
    _same_rows(got, E.sort_rows(np.concatenate(want)), f"tma n={n}")
    assert head == len(got) > n
    _metric_tallies(sim, got, 59)


def _task(name, n, **env):
    import ouzelum_b200
    cfg = ouzelum_b200.task_config(name, n, seed=5, maxEpisodeLength=30, **env)
    return ouzelum_b200.make(seed=5, task=name, num_envs=n, sim_device=DEV, rl_device=DEV, headless=True, cfg=cfg)


@pytest.mark.parametrize("name,early", [("Landing", False), ("Landing", None), ("Landed", None), ("LeeLanded", False),
                                        ("LeeLanded", None), ("Ouzelum", None)])
def test_task_api_and_front_steps(name, early):
    """ozl_landing_step / ozl_lee_landed_step twins (generic and sub-wave) through the task API: the records are those of the
    handle's own post-step state, episode_log() decodes and clears them, and the outputs equal a task without the log."""
    fault = {"enable": True, "mode": "multi", "rotors": [1, 3], "rampSteps": 4} if name in ("Landing", "Ouzelum") else {"enable": True}
    kw = dict(rotorFault=fault, domainRandomization={"enable": True}, asymmetric_observations=True)
    with _kernel_env(early=early):
        env = _task(name, 1500, **kw)
        twin = _task(name, 1500, **kw)
    env.enable_episode_log(4 * 1500)
    mode = env.native_cfg.fault_mode
    want, n_ep = [], 0
    for t in range(90):
        a = _actions(1500, t)
        o1, r1, d1, _ = env.step(a)
        o2, r2, d2, _ = twin.step(a)
        assert torch.equal(o1["obs"], o2["obs"]) and torch.equal(o1["states"], o2["states"]) and torch.equal(r1, r2), t
        assert torch.equal(d1, d2), t
        b = dict(reset=env.reset_buf, progress=env.progress_buf, timeout=env._timeout_u8, ep_ret=env.episode_return_buf)
        want.append(_records_from_state(env.sim, b, t, mode, act_mode=1 if name == "LeeLanded" else 0))
        if t % 30 == 29:
            log = env.episode_log(clear=True)
            w = E.sort_rows(np.concatenate(want))
            want = []
            assert log["dropped"] == 0 and len(log["env"]) == len(w)
            assert torch.equal(log["env"].cpu(), torch.from_numpy(w[:, E.ENV].astype(np.int64)))
            assert torch.equal(log["step"].cpu(), torch.from_numpy(w[:, E.STEP].astype(np.int64)))
            assert torch.equal(log["params"].cpu(), torch.from_numpy(w[:, E.MASS:E.MASS + 7].view(np.float32)))
            assert torch.equal(log["eff"].cpu(), torch.from_numpy(w[:, E.EFF:E.EFF + 4].view(np.float32)))
            assert torch.equal(log["pos"].cpu(), torch.from_numpy(w[:, E.POS:E.POS + 3].view(np.float32)))
            assert torch.equal(log["return"].cpu(), torch.from_numpy(w[:, E.RETURN].view(np.float32)))
            assert torch.equal(log["landed"].cpu(), torch.from_numpy((w[:, E.FLAGS] & E.LANDED) != 0))
            assert torch.equal(log["onset"].cpu(), torch.from_numpy(w[:, E.ONSET].view(np.int32).astype(np.int64)))
            n_ep += len(w)
    assert n_ep > 1500
    sd = env.state_dict()
    assert not any("log" in k for k in sd)                     # the log is not env state
    env.disable_episode_log()
    o1, *_ = env.step(_actions(1500, 99))
    assert env._eplog is None


def test_shards_graph_replay_and_overflow():
    """Two shards give the record set of one handle; a CUDA-graph replay gives the eager steps' set; with a capacity below the
    episode count, head counts every episode and exactly `capacity` rows are written, each a member of the full set."""
    n, h = 4096, 2048
    kw = dict(BASE, **FAULTS[2])
    rows = mf_rows(n, seed=4)
    full, bf, _ = _mk(n, True, rows=rows, **dict(kw, env_id_base=0))
    lo, bl, _ = _mk(h, True, rows=rows[:h].clone(), **dict(kw, env_id_base=0))
    hi, bh, _ = _mk(h, True, rows=rows[h:].clone(), **dict(kw, env_id_base=h))
    gr, bg, _ = _mk(n, True, rows=rows, **dict(kw, env_id_base=0))
    small, bs, _ = _mk(n, True, rows=rows, capacity=1000, **dict(kw, env_id_base=0))
    static_a = torch.zeros(n, 4, device=DEV)
    for s, bb in ((gr, bg), (full, bf), (small, bs)):
        _step(s, bb, static_a)
    _step(lo, bl, static_a[:h].contiguous())
    _step(hi, bh, static_a[h:].contiguous())
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _step(gr, bg, static_a)
    for t in range(100):
        a = _actions(n, t)
        _step(full, bf, a)
        _step(small, bs, a)
        _step(lo, bl, a[:h].contiguous())
        _step(hi, bh, a[h:].contiguous())
        static_a.copy_(a)
        g.replay()
    want, head = _read(full)
    _same_rows(E.sort_rows(np.concatenate([_read(lo)[0], _read(hi)[0]])), want, "shards")
    _same_rows(_read(gr)[0], want, "graph")
    got, shead = _read(small)
    assert shead == head > 1000 and len(got) == 1000
    member = {r.tobytes() for r in want}
    assert all(r.tobytes() in member for r in got)
    # clearing is the caller's zeroing of head: the next records start at row 0 again
    small.head.zero_()
    _step(small, bs, _actions(n, 200))
    k = int(small.head.item())
    assert 0 < k <= n


def test_refusals():
    from ouzelum_b200._lib import OzlEkfLeeArgs, OzlHuskyArgs, lib
    n = 64
    msg = lambda: lib.ozl_last_error().decode()
    sim, b, _ = _mk(n, True, states=False, **BASE)
    assert lib.ozl_rollout(sim._h, 4, b["obs"].data_ptr(), b["rew"].data_ptr(), b["reset"].data_ptr(), b["progress"].data_ptr(),
                           None) != 0 and "episode log" in msg()
    husky = OzlHuskyArgs()
    assert lib.ozl_ekf_lee_landed_step(sim._h, C.byref(OzlEkfLeeArgs()), C.byref(husky), b["obs"].data_ptr(), b["rew"].data_ptr(),
                                       b["reset"].data_ptr(), b["progress"].data_ptr(), None, None, None) != 0 and "episode log" in msg()
    rec, head = sim.records, sim.head
    for args, text in [((rec.data_ptr(), 8, head.data_ptr(), 31), "width 31"), ((rec.data_ptr(), 0, head.data_ptr(), 32), "capacity 0"),
                       ((rec.data_ptr() + 4, 8, head.data_ptr(), 32), "16-byte aligned"), ((rec.data_ptr(), 8, None, 32), "head is NULL")]:
        assert lib.ozl_set_episode_log(sim._h, *args) != 0 and text in msg(), (args, msg())
    # unregistered: the roll-out runs again
    assert lib.ozl_set_episode_log(sim._h, None, 0, None, 32) == 0
    assert lib.ozl_rollout(sim._h, 2, b["obs"].data_ptr(), b["rew"].data_ptr(), b["reset"].data_ptr(), b["progress"].data_ptr(),
                           None) == 0
    for name in ("EKFLeeLanded", "Quadcopter"):
        env = _task(name, 64)
        with pytest.raises(ValueError, match="episode log"):
            env.enable_episode_log(64)


def test_run_episodes():
    """scenarios.run_episodes drains the log often enough to lose nothing, whatever the capacity."""
    from ouzelum_b200 import scenarios
    env = _task("Ouzelum", 512, rotorFault={"enable": True})
    a = torch.zeros(512, 4, device=DEV)
    env.metrics(clear=True)
    out = scenarios.run_episodes(env, lambda obs: a, 100, capacity=512 * 3)
    m = env.metrics().cpu()
    assert out["dropped"] == 0 and len(out["env"]) == int(m[9]) > 512
    assert int(out["length"].sum()) == int(m[10])
    assert bool((out["step"][1:] >= out["step"][:-1]).all())
    assert env._eplog is None
