"""Privileged critic state written by the step kernels (ozl_set_states_output, env.asymmetric_observations): bit-exact against the
CPU reference (tests/states_ref.py), identical on both step kernels, invisible to every other output, and through the task surface
(make(), CUDA graphs, host steps, checkpoints, roll-out storage)."""
import ctypes as C
import os

import pytest
import torch

import states_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROUGH = dict(seed=7, fault_mode=1, dr_enable=1, pomdp_mode=3, pomdp_prob=0.3, noise_sigma=0.15, max_episode_length=40,
             lin_drag=0.05, yaw_km=0.016, env_id_base=123456)


def _mk(n, tma=None, states=True, **kw):
    from ouzelum_b200 import _lib
    from ouzelum_b200.sim import QuadSim
    if "dr_enable" in kw:                                     # all six parameters (default) plus yaw_km
        kw.setdefault("dr", {6: (_lib.DR_UNIFORM, _lib.DR_SCALING, 0.5, 1.5)})
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
    return sim, b, cfg


def _step(sim, b, a):
    sim.step(a, b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"])


def _actions(n, t):
    g = torch.Generator().manual_seed(1000 + t)
    return ((torch.rand(n, 4, generator=g) * 2 - 1) * 0.3).to(DEV)


def _everything(sim, b):
    st = sim.get_state()
    p, f = sim.get_params()
    out = {k: v.clone() for k, v in b.items()}
    out.update({"st_" + k: v for k, v in st.items()}, params=p, fault=f, counts=sim.metrics()[8:16].clone())
    return out


@pytest.mark.parametrize("n", [1, 37, 4099])
def test_generic_kernel_states_equal_reference(n):
    sim, b, cfg = _mk(n, tma=False, **ROUGH)
    ora = R.StatesOracle(cfg.to_dict())
    seen_active = seen_idle = 0
    for t in range(150):
        a = _actions(n, t)
        _step(sim, b, a)
        ora.step(a.cpu())
        s = b["states"].cpu()
        assert torch.equal(b["obs"].cpu(), ora.obs_buf), f"t={t}: obs"
        assert torch.equal(s, ora.states_buf), f"t={t}: states differ in slots {sorted(set((s != ora.states_buf).nonzero()[:, 1].tolist()))}"
        # effectiveness slots: all ones until the env's fault is active, then exactly the faulted rotor carries its effectiveness
        active = (ora.progress_buf - 1) >= ora.fault_onset
        eff = s[:, 17:21]
        assert (eff[~active] == 1).all()
        if active.any():
            rows = active.nonzero()[:, 0]
            assert torch.equal(eff[rows, ora.fault_rotor[rows]], ora.fault_eff[rows])
        seen_active += int(active.sum())
        seen_idle += int((~active).sum())
    assert int(b["timeout"].sum()) >= 0 and seen_active > 0 and (n == 1 or seen_idle > 0)
    assert not torch.equal(b["states"][:, :13], b["obs"]) or n == 1       # pomdp_mode 3: the delivered obs is not the clean one


def test_states_of_non_randomised_parameters_are_exactly_one():
    n = 300
    sim, b, _ = _mk(n, tma=False, seed=3, max_episode_length=20)
    for t in range(25):
        _step(sim, b, _actions(n, t))
    assert (b["states"][:, 21:27] == 1.0).all()
    assert (b["states"][:, 27] == 0.0).all() and (b["states"][:, 17:21] == 1.0).all()


def test_tma_kernel_and_ragged_tail_equal_generic_kernel():
    n = 262144 + 77
    (ta, tb, _), (ga, gb, _) = _mk(n, tma=True, **ROUGH), _mk(n, tma=False, **ROUGH)
    for t in range(30):
        a = _actions(n, t)
        _step(ta, tb, a)
        _step(ga, gb, a)
    x, y = _everything(ta, tb), _everything(ga, gb)
    for k in x:
        assert torch.equal(x[k], y[k]), k
    assert not torch.isnan(tb["states"]).any()


@pytest.mark.parametrize("tma", [False, True])
def test_registering_states_changes_nothing_else(tma):
    n = 262144 + 77 if tma else 4099
    (sa, ba, _), (sb, bb, _) = _mk(n, tma=tma, states=True, **ROUGH), _mk(n, tma=tma, states=False, **ROUGH)
    for t in range(40):
        a = _actions(n, t)
        _step(sa, ba, a)
        _step(sb, bb, a)
    x, y = _everything(sa, ba), _everything(sb, bb)
    del x["states"]
    assert sorted(x) == sorted(y)
    for k in y:
        assert torch.equal(x[k], y[k]), k


@pytest.mark.parametrize("tma", [False, True])
def test_without_sensor_faults_the_state_starts_with_the_observation(tma):
    n = 262144 + 77 if tma else 4099
    kw = dict(ROUGH, pomdp_mode=0)
    sim, b, _ = _mk(n, tma=tma, **kw)
    for t in range(30):
        _step(sim, b, _actions(n, t))
        assert torch.equal(b["states"][:, :13], b["obs"])


def test_shards_equal_the_full_handle():
    n, h = 4096, 2048
    full, bf, _ = _mk(n, tma=False, **dict(ROUGH, env_id_base=0))
    lo, bl, _ = _mk(h, tma=False, **dict(ROUGH, env_id_base=0))
    hi, bh, _ = _mk(h, tma=False, **dict(ROUGH, env_id_base=h))
    for t in range(60):
        a = _actions(n, t)
        _step(full, bf, a)
        _step(lo, bl, a[:h].contiguous())
        _step(hi, bh, a[h:].contiguous())
        assert torch.equal(bf["states"], torch.cat([bl["states"], bh["states"]]))


def test_host_step_writes_the_same_states_as_the_device_step():
    from ouzelum_b200._lib import OzlHostIo, check, lib
    n = 1000
    dev, bd, _ = _mk(n, tma=False, **ROUGH)
    host, bh, _ = _mk(n, tma=False, **ROUGH)
    pin = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt).pin_memory()
    a_h, o_h, r_h, d_h = pin(n, 4), pin(n, 13), pin(n), pin(n, dt=torch.uint8)
    io = OzlHostIo(a_h.data_ptr(), o_h.data_ptr(), r_h.data_ptr(), d_h.data_ptr(), None, bh["reset"].data_ptr(),
                   bh["progress"].data_ptr(), bh["timeout"].data_ptr(), bh["ep_ret"].data_ptr())
    for t in range(50):
        a = _actions(n, t)
        _step(dev, bd, a)
        a_h.copy_(a.cpu())
        check(lib.ozl_step_host_sync(host._h, C.byref(io), torch.cuda.current_stream().cuda_stream))
        assert torch.equal(bd["states"], bh["states"]), t
        assert torch.equal(bd["obs"].cpu(), o_h)


def _task(name, n, **env):
    import ouzelum_b200
    cfg = ouzelum_b200.task_config(name, n, seed=5, maxEpisodeLength=30, asymmetric_observations=True, **env)
    return ouzelum_b200.make(seed=5, task=name, num_envs=n, sim_device=DEV, rl_device=DEV, headless=True, cfg=cfg)


@pytest.mark.parametrize("name", ["Ouzelum", "Lando", "Landing", "Landed", "LeeLanded"])
def test_tasks_deliver_the_kernel_states(name):
    n = 300
    extra = {} if name == "LeeLanded" else dict(rotorFault={"enable": True}, domainRandomization={"enable": True})
    eager, graphed = _task(name, n, **extra), _task(name, n, useCudaGraph=True, **extra)
    assert eager.num_states == 32 and eager.state_space.shape == (32,)
    act_mode = 1 if name == "LeeLanded" else 0
    for t in range(40):
        a = _actions(n, t)
        od, _, _, _ = eager.step(a)
        og, _, _, _ = graphed.step(a)
        s = od["states"]
        assert s.shape == (n, 32) and s.data_ptr() == eager.states_buf.data_ptr()
        assert torch.equal(s.cpu(), R.states_from_task(eager, act_mode)), f"{name} t={t}"
        assert torch.equal(og["states"], s) and torch.equal(og["obs"], od["obs"]), f"{name} t={t}: graph replay != eager"
    assert torch.equal(eager.get_state(), eager.states_buf) and torch.equal(eager.reset()["states"], eager.states_buf)
    if name == "Landed":                                              # flicker model on the delivered observation only
        assert (eager.states_buf[:, :13] != 0).any()


def test_checkpoint_round_trip_keeps_the_states():
    n = 500
    env = _task("Ouzelum", n, rotorFault={"enable": True}, domainRandomization={"enable": True})
    for t in range(15):
        env.step(_actions(n, t))
    sd = env.state_dict()
    assert torch.equal(sd["states_buf"], env.states_buf.cpu())
    env2 = _task("Ouzelum", n, rotorFault={"enable": True}, domainRandomization={"enable": True})
    env2.load_state_dict(sd)
    assert torch.equal(env2.reset()["states"], env.reset()["states"])
    for t in range(15, 35):
        a = _actions(n, t)
        assert torch.equal(env2.step(a)[0]["states"], env.step(a)[0]["states"]), t


def test_refusals():
    from ouzelum_b200 import _lib
    from ouzelum_b200._lib import OzlEkfLeeArgs, OzlHuskyArgs, lib
    sim, b, _ = _mk(64, **ROUGH)
    msg = lambda: lib.ozl_last_error().decode()
    assert lib.ozl_set_states_output(sim._h, b["states"].data_ptr(), 31) != 0 and "OZL_STATES_WIDTH" in msg()
    assert lib.ozl_rollout(sim._h, 4, b["obs"].data_ptr(), b["rew"].data_ptr(), b["reset"].data_ptr(), b["progress"].data_ptr(),
                           None) != 0 and "states" in msg()
    args, husky = OzlEkfLeeArgs(), OzlHuskyArgs()
    assert lib.ozl_ekf_lee_landed_step(sim._h, C.byref(args), C.byref(husky), b["obs"].data_ptr(), b["rew"].data_ptr(),
                                       b["reset"].data_ptr(), b["progress"].data_ptr(), None, None, None) != 0 and "states" in msg()
    sim.set_states_output(None)                                     # unregistered: the roll-out runs again
    sim.rollout(4, b["obs"], b["rew"], b["reset"], b["progress"])
    torch.cuda.synchronize()
    for name in ("EKFLeeLanded", "Quadcopter"):
        with pytest.raises(ValueError, match="asymmetric_observations"):
            _task(name, 64)
    with pytest.raises(ValueError, match="numStates"):
        _task("Ouzelum", 64, numStates=16)
    assert _lib.STATES_WIDTH == 32


def test_graphed_rollout_stores_states_like_eager_collection():
    import ouzelum_b200
    from ouzelum_b200.rollout import GraphedRollout, RecurrentActor, RolloutStorage, collect_rollout, initial_rollout_state
    n, T = 1024, 16

    class MeanActor(RecurrentActor):
        def forward(self, obs, lstm_state, done, action=None):
            mean, std, lstm_state = self.distribution(obs, lstm_state, done)
            logp, ent = self.log_prob_entropy(mean, std, mean)
            return mean, logp, ent, lstm_state
    torch.manual_seed(0)
    actor = MeanActor().to(DEV)
    with torch.no_grad():
        actor.actor_mean.weight.mul_(30.0)
    mk = lambda: _task("Landing", n, rotorFault={"enable": True})
    e_eager, e_graph = mk(), mk()
    s_eager, s_graph = RolloutStorage(T, n, 13, 4, DEV, num_states=32), RolloutStorage(T, n, 13, 4, DEV, num_states=32)
    gro = GraphedRollout(e_graph, actor, s_graph)
    state = initial_rollout_state(e_eager, actor)
    for _ in range(2):
        state = collect_rollout(e_eager, actor, s_eager, state)
    for it in range(3):
        state = collect_rollout(e_eager, actor, s_eager, state)
        gro.run()
        torch.cuda.synchronize()
        for name in ("obs", "states", "actions", "logprobs", "rewards", "dones"):
            assert torch.equal(getattr(s_eager, name), getattr(s_graph, name)), f"rollout {it}: {name}"
    # states[t] belongs to obs[t]: same step, clean observation in front (Landing has no sensor-fault model)
    assert torch.equal(s_eager.states[..., :13], s_eager.obs)
    assert RolloutStorage(T, n, 13, 4, DEV).states is None
