"""Scenario tables (ozl_set_scenarios, X500Task.set_scenarios): an all-NaN table is no table, bit for bit; a mixed table gives the CPU
reference's results (tests/scenario_ref.py) on both step kernels; the pinned conditions do not depend on the policy, follow table
updates into captured graphs, are shard-invariant and survive a checkpoint; invalid tables and unsupported paths are refused."""
import ctypes as C
import math
import os

import pytest
import torch

import scenario_ref as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROUGH = dict(seed=7, fault_mode=1, dr_enable=1, pomdp_mode=3, pomdp_prob=0.3, noise_sigma=0.15, max_episode_length=40,
             target_period=9, lin_drag=0.05, yaw_km=0.016, env_id_base=123456)


def _mk(n, tma=None, rows=None, states=True, **kw):
    from ouzelum_b200 import _lib
    from ouzelum_b200.sim import QuadSim
    if "dr_enable" in kw:                                     # uniform (default) on five parameters, gaussian thrust scale, uniform yaw_km
        kw.setdefault("dr", {5: (_lib.DR_GAUSSIAN, _lib.DR_SCALING, 1.0, 0.05), 6: (_lib.DR_UNIFORM, _lib.DR_SCALING, 0.5, 1.5)})
    old = os.environ.get("OZL_TMA_MIN_TILES")
    if tma is not None:
        os.environ["OZL_TMA_MIN_TILES"] = "1" if tma else "0"     # read once per handle at ozl_create
    try:
        cfg = _lib.default_cfg(n, **kw)
        sim = QuadSim(cfg, DEV)
    finally:
        if old is None:
            os.environ.pop("OZL_TMA_MIN_TILES", None)
        else:
            os.environ["OZL_TMA_MIN_TILES"] = old
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


def _actions(n, t, scale=0.3, seed=1000):
    g = torch.Generator().manual_seed(seed + t)
    return ((torch.rand(n, 4, generator=g) * 2 - 1) * scale).to(DEV)


def _everything(sim, b):
    st = sim.get_state()
    p, f = sim.get_params()
    out = {k: v.clone() for k, v in b.items()}
    m = sim.metrics()
    out.update({"st_" + k: v for k, v in st.items()}, params=p, fault=f, counts=torch.cat([m[2:3], m[8:16]]).clone())
    return out


@pytest.mark.parametrize("n,tma", [(4099, False), (262144 + 77, True), (37, False)])
def test_all_nan_table_is_no_table(n, tma):
    (sa, ba, _), (sb, bb, _) = _mk(n, tma=tma, rows=S.empty(n), **ROUGH), _mk(n, tma=tma, **ROUGH)
    for t in range(150):
        a = _actions(n, t)
        _step(sa, ba, a)
        _step(sb, bb, a)
    x, y = _everything(sa, ba), _everything(sb, bb)
    assert int(y["counts"][2]) > 0 and int(y["counts"][7]) > 0          # episodes finished, rotor faults were active
    for k in y:
        assert torch.equal(x[k], y[k]), k


@pytest.mark.parametrize("n,tma", [(4099, False), (4099, True), (300, False)])
def test_kernel_equals_the_reference_on_a_mixed_table(n, tma):
    from ouzelum_b200 import _lib
    cfg = _lib.default_cfg(n, **dict(ROUGH, dr={5: (_lib.DR_GAUSSIAN, _lib.DR_SCALING, 1.0, 0.05),
                                               6: (_lib.DR_UNIFORM, _lib.DR_SCALING, 0.5, 1.5)}))
    rows = S.mixed_rows(n, cfg.to_dict(), seed=5)
    sim, b, cfg = _mk(n, tma=tma, rows=rows, **ROUGH)
    ora = S.ScenarioOracle(cfg.to_dict(), rows)
    full = torch.arange(n) % 3 == 0
    eff_seen = 0
    for t in range(150):
        a = _actions(n, t)
        _step(sim, b, a)
        ora.step(a.cpu())
        for k, o in (("obs", ora.obs_buf), ("rew", ora.rew_buf), ("reset", ora.reset_buf), ("progress", ora.progress_buf),
                     ("states", ora.states_buf)):
            assert torch.equal(b[k].cpu(), o), f"t={t}: {k}"
        s = b["states"].cpu()
        # the states row carries the pinned body parameters and, once the pinned fault is active, the pinned effectiveness
        assert torch.equal(s[full, 21], torch.clamp(rows[full, S.MASS] / torch.tensor(cfg.mass), -5, 5))
        act = full & (ora.progress_buf - 1 >= ora.fault_onset) & (rows[:, S.ROTOR] >= 0)
        if act.any():
            idx = act.nonzero()[:, 0]
            assert torch.equal(s[idx, 17 + rows[idx, S.ROTOR].long()], rows[idx, S.EFF])
            eff_seen += len(idx)
    st = sim.get_state()
    assert torch.equal(st["root"].cpu(), ora.root) and torch.equal(st["target"].cpu(), ora.target)
    assert eff_seen > 0


def _same(x, y):
    """Equal, NaN where NaN."""
    return torch.equal(torch.isnan(x), torch.isnan(y)) and torch.equal(torch.nan_to_num(x), torch.nan_to_num(y))


def _pinned_check(sim, b, rows, full):
    """After the step: apply the pending resets and compare the pinned groups of the resetting envs with their rows."""
    sim.apply_resets(b["reset"])
    st, (p, f) = sim.get_state(), sim.get_params()
    r = (b["reset"] != 0).cpu() & full
    root, tgt, p, f = st["root"].cpu()[r], st["target"].cpu()[r], p.cpu()[r], f.cpu()[r]
    rr = rows[r]
    assert torch.equal(root, rr[:, 0:13])
    assert torch.equal(tgt, rr[:, S.TARGET:S.TARGET + 3])
    assert torch.equal(p[:, [0, 1, 2, 3, 4, 5, 7]], rr[:, S.MASS:S.YAW_KM + 1]) and torch.equal(p[:, 6], rr[:, S.EFF])
    none = rr[:, S.ROTOR] < 0
    assert torch.equal(f[:, 0][~none], rr[:, S.ROTOR][~none].int()) and torch.equal(f[:, 1][~none] & 0x1FFFFFFF, rr[:, S.ONSET][~none].int())
    assert ((f[:, 1][none] & 0x1FFFFFFF) == S.FAULT_NEVER).all()
    return int(r.sum())


def test_pinned_conditions_do_not_depend_on_the_policy():
    n = 999
    sims = []
    from ouzelum_b200 import _lib
    rows = S.mixed_rows(n, _lib.default_cfg(n, **ROUGH).to_dict(), seed=9)
    full = torch.arange(n) % 3 == 0
    for seed in (1, 2):
        sim, b, _ = _mk(n, tma=False, rows=rows, **ROUGH)
        checked = 0
        for t in range(120):
            _step(sim, b, _actions(n, t, scale=0.3 * seed, seed=seed * 10000))
            checked += _pinned_check(sim, b, rows, full)
        sims.append((sim, b))
        assert checked > 100
    assert not torch.equal(sims[0][1]["reset"], sims[1][1]["reset"]) or not torch.equal(sims[0][1]["obs"], sims[1][1]["obs"])


def _task(name, n, **env):
    import ouzelum_b200
    cfg = ouzelum_b200.task_config(name, n, seed=5, maxEpisodeLength=30, **env)
    return ouzelum_b200.make(seed=5, task=name, num_envs=n, sim_device=DEV, rl_device=DEV, headless=True, cfg=cfg)


@pytest.mark.parametrize("name", ["Landing", "Landed", "LeeLanded"])
def test_landing_family_honours_the_table(name):
    n = 300
    fault = name != "LeeLanded"
    env = _task(name, n, **(dict(rotorFault={"enable": True}) if fault else {}), domainRandomization={"enable": True})
    cfg = env.native_cfg.to_dict()
    rows = S.mixed_rows(n, cfg, seed=2)
    assert torch.isnan(rows[:, S.TARGET]).all() and (fault == (not torch.isnan(rows[:, S.ROTOR]).all()))
    bad = rows.clone()
    bad[0, S.TARGET:S.TARGET + 3] = torch.tensor([0.0, 0.0, 1.0])
    with pytest.raises(ValueError, match="target"):
        env.set_scenarios(bad)
    if not fault:
        bad = rows.clone()
        bad[0, S.ROTOR:S.EFF + 1] = torch.tensor([1.0, 3.0, 0.5])
        with pytest.raises(ValueError, match="fault"):
            env.set_scenarios(bad)
    env.set_scenarios(rows.to(DEV))
    full = torch.arange(n) % 3 == 0
    checked = 0
    for t in range(80):
        env.step(_actions(n, t))
        env.sim.apply_resets(env.reset_buf)
        st, (p, f) = env.sim.get_state(), env.sim.get_params()
        r = (env.reset_buf != 0).cpu() & full
        assert torch.equal(st["root"].cpu()[r], rows[r, 0:13])
        assert torch.equal(p.cpu()[r][:, [0, 1, 2, 3, 4, 5, 7]], rows[r, S.MASS:S.YAW_KM + 1])
        if fault:
            fr = f.cpu()[r]
            some = rows[r, S.ROTOR] >= 0
            assert torch.equal(fr[some, 0], rows[r][some, S.ROTOR].int()) and torch.equal(p.cpu()[r][:, 6], rows[r, S.EFF])
        checked += int(r.sum())
    assert checked > 0


def test_graph_replay_follows_table_updates():
    from ouzelum_b200 import _lib
    n = 600
    cfg = _lib.default_cfg(n, **ROUGH).to_dict()
    r1, r2 = S.mixed_rows(n, cfg, seed=1), S.mixed_rows(n, cfg, seed=2)
    full = torch.arange(n) % 3 == 0
    eager = _task("Ouzelum", n, rotorFault={"enable": True}, domainRandomization={"enable": True})
    graphed = _task("Ouzelum", n, rotorFault={"enable": True}, domainRandomization={"enable": True}, useCudaGraph=True)
    for env in (eager, graphed):
        env.set_scenarios(r1)
    for t in range(60):
        if t == 20:
            assert graphed._graph is not None
            for env in (eager, graphed):
                env.set_scenarios(r2)          # same address, new contents: the captured graph sees them
            assert graphed._graph is not None
        a = _actions(n, t)
        oe, og = eager.step(a)[0]["obs"], graphed.step(a)[0]["obs"]
        assert torch.equal(oe, og), t
        if t >= 20:
            graphed.sim.apply_resets(graphed.reset_buf)
            r = (graphed.reset_buf != 0).cpu() & full
            assert torch.equal(graphed.sim.get_state()["root"].cpu()[r], r2[r, 0:13]), t


def test_graphed_rollout_follows_table_updates():
    from ouzelum_b200 import _lib
    from ouzelum_b200.rollout import GraphedRollout, RecurrentActor, RolloutStorage, collect_rollout, initial_rollout_state
    n, T = 1024, 16

    class MeanActor(RecurrentActor):                          # deterministic actions: eager and graphed passes see the same ones
        def forward(self, obs, lstm_state, done, action=None):
            mean, std, lstm_state = self.distribution(obs, lstm_state, done)
            logp, ent = self.log_prob_entropy(mean, std, mean)
            return mean, logp, ent, lstm_state
    torch.manual_seed(0)
    actor = MeanActor().to(DEV)
    with torch.no_grad():
        actor.actor_mean.weight.mul_(30.0)
    mk = lambda: _task("Ouzelum", n, rotorFault={"enable": True})
    e_eager, e_graph = mk(), mk()
    cfg = e_eager.native_cfg.to_dict()
    tables = [S.mixed_rows(n, cfg, seed=s) for s in (11, 12, 13)]
    for env in (e_eager, e_graph):
        env.set_scenarios(tables[0])
    s_eager, s_graph = RolloutStorage(T, n, 13, 4, DEV), RolloutStorage(T, n, 13, 4, DEV)
    gro = GraphedRollout(e_graph, actor, s_graph)
    state = initial_rollout_state(e_eager, actor)
    for _ in range(2):
        state = collect_rollout(e_eager, actor, s_eager, state)
    for it in range(3):
        for env in (e_eager, e_graph):
            env.set_scenarios(tables[it])
        state = collect_rollout(e_eager, actor, s_eager, state)
        gro.run()
        torch.cuda.synchronize()
        for name in ("obs", "actions", "rewards", "dones"):
            assert torch.equal(getattr(s_eager, name), getattr(s_graph, name)), f"rollout {it}: {name}"
        assert int(s_graph.dones.sum()) > 0


def test_shards_equal_the_full_handle():
    from ouzelum_b200 import _lib
    n, h = 4096, 2048
    rows = S.mixed_rows(n, _lib.default_cfg(n, **ROUGH).to_dict(), seed=4)
    full, bf, _ = _mk(n, tma=False, rows=rows, **dict(ROUGH, env_id_base=0))
    lo, bl, _ = _mk(h, tma=False, rows=rows[:h].clone(), **dict(ROUGH, env_id_base=0))
    hi, bh, _ = _mk(h, tma=False, rows=rows[h:].clone(), **dict(ROUGH, env_id_base=h))
    for t in range(80):
        a = _actions(n, t)
        _step(full, bf, a)
        _step(lo, bl, a[:h].contiguous())
        _step(hi, bh, a[h:].contiguous())
        for k in ("obs", "rew", "reset", "states"):
            assert torch.equal(bf[k], torch.cat([bl[k], bh[k]])), (t, k)


def test_refusals_and_validation():
    from ouzelum_b200 import _lib
    from ouzelum_b200._lib import OzlEkfLeeArgs, OzlHuskyArgs, lib
    n = 64
    sim, b, _ = _mk(n, states=False, **ROUGH)
    msg = lambda: lib.ozl_last_error().decode()
    ok = S.mixed_rows(n, sim.cfg.to_dict(), seed=1)
    sim.set_scenarios(ok)
    assert lib.ozl_rollout(sim._h, 4, b["obs"].data_ptr(), b["rew"].data_ptr(), b["reset"].data_ptr(), b["progress"].data_ptr(),
                           None) != 0 and "scenario" in msg()
    args, husky = OzlEkfLeeArgs(), OzlHuskyArgs()
    assert lib.ozl_ekf_lee_landed_step(sim._h, C.byref(args), C.byref(husky), b["obs"].data_ptr(), b["rew"].data_ptr(),
                                       b["reset"].data_ptr(), b["progress"].data_ptr(), None, None, None) != 0 and "scenario" in msg()
    host = ok.contiguous()
    assert lib.ozl_set_scenarios(sim._h, host.data_ptr(), 31, None) != 0 and "OZL_SCENARIO_WIDTH" in msg()

    def bad(edit, text, **cfg_over):
        s = sim
        if cfg_over:
            s = _mk(n, states=False, **dict(ROUGH, **cfg_over))[0]
        r = S.empty(n)
        edit(r)
        with pytest.raises(ValueError, match=text):
            s.set_scenarios(r)

    def put(sl, vals):
        def f(r):
            r[3, sl] = torch.tensor(vals, dtype=torch.float32)
        return f
    bad(put(slice(26, 27), [0.0]), "reserved slot 26")
    bad(put(slice(0, 3), [1.0, math.nan, 1.0]), "position group must be all NaN or all set")
    bad(put(slice(7, 10), [1.0, math.inf, 1.0]), "linear velocity group has a non-finite")
    bad(put(slice(3, 7), [0.0, 0.0, 0.0, 1.001]), "not unit")
    bad(put(slice(13, 16), [0.0, 0.0, 1.0]), "target_fixed", target_fixed=1)
    bad(put(slice(16, 19), [1.0, 0.0, 0.5]), "rotorFault.enable", fault_mode=0)
    bad(put(slice(16, 19), [4.0, 0.0, 0.5]), "rotor")
    bad(put(slice(16, 19), [1.5, 0.0, 0.5]), "rotor")
    bad(put(slice(16, 19), [1.0, 2.5, 0.5]), "onset")
    bad(put(slice(16, 19), [1.0, float(1 << 24), 0.5]), "onset")
    bad(put(slice(16, 19), [1.0, -1.0, 0.5]), "onset")
    bad(put(slice(16, 19), [1.0, 3.0, 1.5]), "effectiveness")
    bad(put(slice(19, 20), [0.0]), "mass / inertia")
    bad(put(slice(22, 23), [1e-38]), "mass / inertia")
    bad(put(slice(23, 24), [0.0]), "arm")
    bad(put(slice(24, 25), [-0.1]), "thrust_scale")
    bad(put(slice(25, 26), [math.inf]), "yaw_km group has a non-finite")
    sim.set_scenarios(S.mixed_rows(n, sim.cfg.to_dict(), seed=2))       # the failed calls left the table registered and usable
    sim.set_scenarios(None)                                             # unregistered: the roll-out runs again
    sim.rollout(4, b["obs"], b["rew"], b["reset"], b["progress"])
    torch.cuda.synchronize()
    for name in ("EKFLeeLanded", "Quadcopter"):
        env = _task(name, 64)
        with pytest.raises(ValueError, match="scenario"):
            env.set_scenarios(S.empty(64))
    with pytest.raises(ValueError):
        sim.set_scenarios(S.empty(n + 1))
    assert _lib.SCENARIO_WIDTH == 32


def test_checkpoint_round_trip_with_a_table():
    n = 500
    kw = dict(rotorFault={"enable": True}, domainRandomization={"enable": True}, asymmetric_observations=True)
    env = _task("Ouzelum", n, **kw)
    rows = S.mixed_rows(n, env.native_cfg.to_dict(), seed=8)
    env.set_scenarios(rows)
    for t in range(25):
        env.step(_actions(n, t))
    sd = env.state_dict()
    assert _same(sd["scenarios"], rows)
    env2 = _task("Ouzelum", n, **kw)
    env2.load_state_dict(sd)
    assert _same(env2.scenarios, rows)
    for t in range(25, 80):
        a = _actions(n, t)
        o1, r1, d1, _ = env.step(a)
        o2, r2, d2, _ = env2.step(a)
        assert torch.equal(o1["obs"], o2["obs"]) and torch.equal(o1["states"], o2["states"]), t
        assert torch.equal(r1, r2) and torch.equal(d1, d2), t


def test_evaluate_counts_episodes_on_the_device():
    from ouzelum_b200 import scenarios
    n = 256
    env = _task("Ouzelum", n, rotorFault={"enable": True})
    env.set_scenarios(scenarios.fault_grid(n, rotors=[-1, 0, 1, 2, 3], onsets=[0, 10], effectiveness=[0.0, 0.5]))
    res = scenarios.evaluate(env, lambda obs: torch.zeros(n, 4, device=DEV), 100)
    assert res["episodes"].device.type == "cuda" and int(res["episodes"].sum()) > 0
    assert (res["survived"] <= res["episodes"]).all()
    m = env.metrics().cpu()
    assert int(res["episodes"].sum()) == int(m[9]) and int(res["survived"].sum()) == int(m[11])
    assert float(res["return_sum"].sum()) == pytest.approx(float(m[1]), rel=1e-4)
