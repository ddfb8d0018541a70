"""The episode-metrics vector (ozl_metrics_read) of every step-kernel path against the exact tallies of the CPU oracle
(tests/metrics_ref.py), all 16 slots under one rule: slots 2-15 equal to the reference (3-7 zero), slots 0-1 within the worst
case of float64 summation of their float32 terms in any order.

Three separately written reductions feed the vector: `block_epilogue<128>` (generic step, its scenario / states twins, the
one-launch vehicle and Lee steps, the ragged tail of the TMA kernel and the last step of a roll-out), `block_epilogue<96>`
(the fused EKFLeeLanded step), the per-CTA reduction of the persistent TMA kernel, and the roll-out's own reduction of its
intermediate steps.  The sizes put partial warps, partial CTAs, several tiles per persistent CTA and ragged tails under test;
every case asserts that the events it is about did occur, so that none passes with empty slots."""
import os

import numpy as np
import pytest
import torch

from metrics_ref import (CRASH_DIST, CRASH_Z, EPISODES, FAULT_STEPS, LANDED, RESETS, TIMEOUTS, MetricsOracle, assert_metrics,
                         with_metrics)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# rotor faults, domain randomisation, flicker + observation noise, short episodes, crash thresholds that the spawn box and the
# targets reach within a few dozen steps: time-outs, both crash causes, fault-active steps and resets all occur
EVENTFUL = dict(fault_mode=1, dr_enable=1, pomdp_mode=3, pomdp_prob=0.3, noise_sigma=0.15, max_episode_length=12, die_z=1.1,
                die_dist=6.0)


def _bufs(n):
    return dict(obs=torch.zeros(n, 13, device=DEV), rew=torch.zeros(n, device=DEV),
                reset=torch.ones(n, dtype=torch.int64, device=DEV), progress=torch.zeros(n, dtype=torch.int64, device=DEV),
                timeout=torch.zeros(n, dtype=torch.uint8, device=DEV), ep_ret=torch.zeros(n, device=DEV))


def _args(b):
    return b["obs"], b["rew"], b["reset"], b["progress"], b["timeout"], b["ep_ret"]


def _sim(n, tma=None, **kw):
    """QuadSim and its cfg.  tma: None = the default kernel selection, True = the persistent TMA kernel from one whole tile on,
    False = never (OZL_TMA_MIN_TILES is read once per handle, at ozl_create)."""
    from ouzelum_b200 import _lib
    from ouzelum_b200.sim import QuadSim
    cfg = _lib.default_cfg(n, **kw)
    old = os.environ.get("OZL_TMA_MIN_TILES")
    if tma is None:
        os.environ.pop("OZL_TMA_MIN_TILES", None)
    else:
        os.environ["OZL_TMA_MIN_TILES"] = "1" if tma else "0"
    try:
        return QuadSim(cfg, DEV), cfg
    finally:
        if old is None:
            os.environ.pop("OZL_TMA_MIN_TILES", None)
        else:
            os.environ["OZL_TMA_MIN_TILES"] = old


def _in_step(reset, progress, ora, tag):
    """The device env step and the oracle's are still the same (else a metrics difference would say nothing about the reduction)."""
    assert torch.equal(reset.cpu(), ora.reset_buf), f"{tag}: reset flags left the oracle"
    assert torch.equal(progress.cpu(), ora.progress_buf), f"{tag}: progress left the oracle"


def _place_on(sim, ora, envs, point=None):
    """Put `envs` at rest on their stored target (or on `point`), in the handle and in the oracle."""
    st = sim.get_state()
    root = st["root"].cpu()
    assert torch.equal(root, ora.root)
    root[envs, 0:3] = st["target"].cpu()[envs] if point is None else torch.tensor(point)
    root[envs, 7:13] = 0.0
    sim.set_state(root=root)
    ora.root = root.clone()


@pytest.mark.parametrize("path", ["step", "wrench", "host"])
@pytest.mark.parametrize("n", [1, 31, 33, 127, 129, 4099])
def test_generic_step_kernel_metrics(n, path):
    """`block_epilogue<128>` with partial warps (1, 31, 33, 4099) and partial CTAs (127, 129, 4099), through ozl_step,
    ozl_step_wrench with a caller target, and the zero-copy ozl_step_host."""
    tag = f"{path} n={n}"
    sim, cfg = _sim(n, seed=5, env_id_base=1000, **EVENTFUL)
    ora = MetricsOracle(cfg.to_dict())
    b = _bufs(n)
    g = torch.Generator().manual_seed(n)
    hover = float(np.float32(2.0643077 * 9.81))
    if path == "host":
        pin = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt).pin_memory()
        h_act, h_obs, h_rew, h_done = pin(n, 4), pin(n, 13), pin(n), pin(n, dt=torch.uint8)
    for t in range(48):
        if path == "wrench":
            w = torch.cat([hover * (0.6 + 0.8 * torch.rand(n, 1, generator=g)), torch.randn(n, 3, generator=g) * 0.05], 1)
            tgt = torch.rand(n, 3, generator=g) * torch.tensor([6.0, 6.0, 1.0]) + torch.tensor([-3.0, -3.0, 1.0])
            sim.step_wrench(w.to(DEV), tgt.to(DEV), *_args(b))
            ora.step(w, target_in=tgt, act_mode=1)
        else:
            a = (torch.rand(n, 4, generator=g) * 2 - 1) * 0.5
            if path == "host":
                h_act.copy_(a)
                sim.step_host(h_act, h_obs, h_rew, h_done, b["reset"], b["progress"], b["timeout"], b["ep_ret"])
                torch.cuda.synchronize()          # the kernel reads the pinned actions in place
            else:
                sim.step(a.to(DEV), *_args(b))
            ora.step(a)
        _in_step(b["reset"], b["progress"], ora, f"{tag} t={t}")
    assert_metrics(sim.metrics(), ora, tag)
    c = ora.counts
    assert c[EPISODES] > 0 and c[TIMEOUTS] > 0 and c[RESETS] > 0, c
    if path != "wrench":                          # wrench actuation never applies a rotor fault
        assert c[FAULT_STEPS] > 0, c
    if n > 1:                                     # a single env times out in every episode of this run
        assert c[CRASH_DIST] + c[CRASH_Z] > 0 and (path == "wrench" or min(c[CRASH_DIST], c[CRASH_Z]) > 0), c


@pytest.mark.parametrize("tma", [False, True], ids=["generic", "tma"])
@pytest.mark.parametrize("twin", ["scenarios", "states", "both"])
def test_scenario_and_states_kernel_twins_metrics(twin, tma):
    """The step kernels instantiated with a scenario table and / or the privileged-state output, generic and persistent TMA."""
    from scenario_ref import ScenarioOracle, mixed_rows
    n = 1001                                      # 7 whole tiles + a 105-env tail
    sim, cfg = _sim(n, tma=tma, seed=8, **EVENTFUL)
    if twin == "states":
        ora = MetricsOracle(cfg.to_dict())
    else:
        rows = mixed_rows(n, cfg.to_dict(), seed=3)
        ora = with_metrics(ScenarioOracle)(cfg.to_dict(), rows)
        sim.set_scenarios(rows)
    if twin != "scenarios":
        states = torch.zeros(n, 32, device=DEV)
        sim.set_states_output(states)
    b = _bufs(n)
    g = torch.Generator().manual_seed(9)
    for t in range(40):
        a = (torch.rand(n, 4, generator=g) * 2 - 1) * 0.5
        sim.step(a.to(DEV), *_args(b))
        ora.step(a)
        _in_step(b["reset"], b["progress"], ora, f"{twin} t={t}")
    assert_metrics(sim.metrics(), ora, f"{twin} tma={tma}")
    c = ora.counts
    assert min(c[EPISODES], c[TIMEOUTS], c[CRASH_DIST], c[CRASH_Z], c[FAULT_STEPS]) > 0, c


@pytest.mark.parametrize("tail", [77, 0], ids=["ragged", "whole_tiles"])
def test_tma_kernel_several_tiles_per_persistent_cta(tail):
    """The persistent TMA kernel accumulates each CTA's metrics over all of its tiles and reduces once: two tiles per CTA and
    more, with and without the one-block tail launch."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * (sms * 5) * 128 + tail               # 5 persistent CTAs per SM
    sim, cfg = _sim(n, tma=True, seed=21, fault_mode=1, dr_enable=1, max_episode_length=6, die_z=1.1, die_dist=6.0)
    ora = MetricsOracle(cfg.to_dict())
    b = _bufs(n)
    g = torch.Generator().manual_seed(4)
    for t in range(12):
        a = (torch.rand(n, 4, generator=g) * 2 - 1) * 0.5
        sim.step(a.to(DEV), *_args(b))
        ora.step(a)
        _in_step(b["reset"], b["progress"], ora, f"n={n} t={t}")
    assert_metrics(sim.metrics(), ora, f"n={n}")
    c = ora.counts
    assert min(c[EPISODES], c[TIMEOUTS], c[CRASH_DIST], c[CRASH_Z], c[FAULT_STEPS]) > 0, c


@pytest.mark.parametrize("tma", [False, True], ids=["generic", "tma"])
def test_landed_episodes_on_the_plain_step(tma):
    """Slot 2 from the landing detector of the plain rotor step: half of the envs are put on their target early in every
    episode, so that episodes end with the landed flag set."""
    n = 4099
    sim, cfg = _sim(n, tma=tma, seed=4, target_fixed=1, land_cutoff=0.2, max_episode_length=5)
    ora = MetricsOracle(cfg.to_dict())
    b = _bufs(n)
    on = torch.arange(n) % 2 == 0
    g = torch.Generator().manual_seed(6)
    for t in range(16):
        if t % 4 == 1:                            # 4-step episodes start at 0, 4, 8, 12
            _place_on(sim, ora, on)
        a = torch.rand(n, 4, generator=g) * 2 - 1
        sim.step(a.to(DEV), *_args(b))
        ora.step(a)
        _in_step(b["reset"], b["progress"], ora, f"t={t}")
    m = sim.metrics().cpu()
    assert int(m[LANDED]) == ora.mlanded, f"slot 2 = {float(m[LANDED])}, landed episodes of the oracle {ora.mlanded}"
    assert ora.mlanded >= int(on.sum()) * 3, ora.mlanded
    assert_metrics(m, ora, f"landing tma={tma}")


def _load(ora, env, t):
    """Adopt the task's device state (the landed flag travels in bit 31 of the onset word)."""
    st = env.sim.get_state()
    params, fault = env.sim.get_params()
    ora.load(st["root"].cpu().numpy(), st["thrust"].cpu().numpy(), st["target"].cpu().numpy(), st["ep_ret"].cpu().numpy(),
             params.cpu().numpy(), fault.cpu().numpy(), env.reset_buf.cpu().numpy(), env.progress_buf.cpu().numpy(), t)


@pytest.mark.parametrize("task", ["Landing", "Landed", "LeeLanded"])
def test_vehicle_and_lee_one_launch_steps_metrics(task):
    """FRONT_VEHICLE (`ozl_landing_step`: Landing, Landed) and FRONT_LEE (`ozl_lee_landed_step`: LeeLanded), the producers of
    slot 2 besides the fused estimator step.  The oracle adopts the device state before every step and takes the vehicle's
    target (and for LeeLanded the kernel's wrench and the controller target as the detector point)."""
    import ouzelum_b200
    n = 3001
    env = ouzelum_b200.make(seed=13, task=task, num_envs=n, sim_device=DEV, rl_device=DEV, headless=True,
                            cfg=ouzelum_b200.task_config(task, n, seed=13, maxEpisodeLength=8, rotorFault={"enable": True}))
    ora = MetricsOracle(env.native_cfg.to_dict())
    lee = task == "LeeLanded"
    hover_point = [0.0, 0.0, 1.0]                 # LeeLanded's controller target (lee_landed.py:299-302)
    on = torch.arange(n) % 2 == 0
    g = torch.Generator().manual_seed(2)
    for t in range(30):
        _load(ora, env, t)
        if t % 7 == 1 and task != "Landing":      # 7-step episodes start at 0, 7, 14, 21, 28
            _place_on(env.sim, ora, on, hover_point if lee else None)
        a = torch.rand(n, 4, generator=g) * 2 - 1
        env.step(a.to(DEV))
        tgt = env.husky.target.cpu()
        if lee:
            ora.step(env._wrench.cpu(), target_in=tgt, act_mode=1, det_target=torch.tensor(hover_point))
        else:
            ora.step(a, target_in=tgt)
        _in_step(env.reset_buf, env.progress_buf, ora, f"{task} t={t}")
        assert torch.equal(env.rew_buf.cpu(), ora.rew_buf), f"{task} t={t}: reward left the oracle"
    assert_metrics(env.metrics(), ora, task)
    c = ora.counts
    assert c[EPISODES] > 0 and c[TIMEOUTS] > 0, c
    if task != "Landing":                         # Landing has no landing detector
        assert c[LANDED] >= int(on.sum()) * 3, c


@pytest.mark.parametrize("n", [31, 960, 4099])
def test_fused_estimator_step_metrics(n):
    """`block_epilogue<96>` of the one-launch EKFLeeLanded step: n = 31 (one partial CTA, no covariance tensor map), 960 (whole
    96-env CTAs, tensor map), 4099 (plain-load fallback, partial CTA).  Envs are put on their target during the estimator
    warm-up (no landing flag may be raised then) and after it."""
    import ouzelum_b200
    conv = 3
    env = ouzelum_b200.make(seed=12, task="EKFLeeLanded", num_envs=n, sim_device=DEV, rl_device=DEV, headless=True,
                            cfg=ouzelum_b200.task_config("EKFLeeLanded", n, seed=12, ConvergenceTime=conv, maxEpisodeLength=6,
                                                         domainRandomization={"enable": True}))
    assert env.fused and env.fused_step
    ora = MetricsOracle(env.native_cfg.to_dict())
    assert ora.cfg["wrench_warmup_steps"] == conv and ora.cfg["land_cutoff"] > 0
    on = torch.arange(n) % 2 == 0
    a = torch.zeros(n, 4, device=DEV)
    for t in range(20):
        _load(ora, env, t)
        if t % 5 == 1:                            # 5-step episodes start at 0, 5, 10, 15; step 1 is inside the warm-up
            _place_on(env.sim, ora, on)
        env.step(a)
        ora.step(env._wrench.cpu(), target_in=env.husky.target.cpu(), act_mode=1)
        _in_step(env.reset_buf, env.progress_buf, ora, f"n={n} t={t}")
        if t < conv:
            _, fault = env.sim.get_params()
            assert not bool((fault[:, 1] < 0).any()), f"t={t}: landing flag raised during the warm-up"
    assert_metrics(env.metrics(), ora, f"EKFLeeLanded n={n}")
    c = ora.counts
    assert c[EPISODES] > 0 and c[RESETS] > n and c[LANDED] >= int(on.sum()), c


@pytest.mark.parametrize("landing", [False, True], ids=["no_cutoff", "land_cutoff"])
@pytest.mark.parametrize("K", [1, 2, 33])
def test_rollout_metrics_equal_k_steps(K, landing):
    """`ozl_rollout(K)` adds to the vector what K single steps add: its intermediate steps go through the kernel's own
    reduction, the last through `block_epilogue<128>`.  With the landing detector, episodes flagged before the roll-out end
    at its first step."""
    from oracle import philox as px
    n, seed = 777, 99
    kw = dict(target_fixed=1, land_cutoff=0.2) if landing else dict(dr_enable=1, die_z=1.1, die_dist=6.0)
    sim, cfg = _sim(n, seed=seed, fault_mode=1, max_episode_length=5, **kw)
    ora = MetricsOracle(cfg.to_dict())
    b = _bufs(n)
    ids = np.arange(n)

    def act(t):                                   # the roll-out's in-kernel actions: 2u - 1 from the P_ACTION stream
        return torch.from_numpy(np.stack([np.float32(2.0) * px.u01(x) - np.float32(1.0)
                                          for x in px.draw(seed, ids, t, px.P_ACTION)], -1))
    on = torch.arange(n) % 2 == 0
    pre = 4                                       # the first episode times out at step 3
    for t in range(pre):
        if t == 1 and landing:
            _place_on(sim, ora, on)
        a = act(t)
        sim.step(a.to(DEV), *_args(b))
        ora.step(a)
    sim.rollout(K, b["obs"], b["rew"], b["reset"], b["progress"])
    for t in range(pre, pre + K):
        ora.step(act(t))
    _in_step(b["reset"], b["progress"], ora, f"K={K}")
    assert torch.equal(b["obs"].cpu(), ora.obs_buf) and sim.step_count == pre + K
    assert_metrics(sim.metrics(), ora, f"rollout K={K} landing={landing}")
    c = ora.counts
    assert c[EPISODES] > 0 and c[FAULT_STEPS] > 0, c
    if landing:
        assert c[LANDED] >= int(on.sum()), c


def _eventful_actions(n, seed):
    g = torch.Generator().manual_seed(seed)
    return lambda: (torch.rand(n, 4, generator=g) * 2 - 1) * 0.5


def test_clearing_reads_sum_to_the_uncleared_vector():
    """Reading with clear=1 every j steps and summing the reads gives the vector of a twin handle that was never cleared."""
    n, j, steps = 1000, 3, 40
    sim, cfg = _sim(n, seed=3, **EVENTFUL)
    twin, _ = _sim(n, seed=3, **EVENTFUL)
    ora = MetricsOracle(cfg.to_dict())
    b, bt = _bufs(n), _bufs(n)
    nxt = _eventful_actions(n, 1)
    reads = []
    for t in range(steps):
        a = nxt()
        sim.step(a.to(DEV), *_args(b))
        twin.step(a.to(DEV), *_args(bt))
        ora.step(a)
        if t % j == j - 1:
            reads.append(sim.metrics(clear=True).cpu().numpy())
    reads.append(sim.metrics(clear=True).cpu().numpy())
    assert not sim.metrics().cpu().numpy().any(), "a clearing read left something behind"
    total, whole = np.sum(reads, axis=0), twin.metrics().cpu().numpy()
    assert np.array_equal(total[2:], whole[2:])
    assert_metrics(total, ora, "sum of clearing reads")
    assert_metrics(whole, ora, "uncleared twin")
    assert min(ora.counts[EPISODES], ora.counts[CRASH_Z], ora.counts[FAULT_STEPS]) > 0


def test_clearing_read_captured_in_a_cuda_graph():
    """The pattern of a timed benchmark: j steps and one clearing read captured in a CUDA graph, replayed; the reads sum to the
    vector of an eager twin."""
    n, j, replays = 1000, 3, 10
    sim, cfg = _sim(n, seed=3, **EVENTFUL)
    twin, _ = _sim(n, seed=3, **EVENTFUL)
    ora = MetricsOracle(cfg.to_dict())
    b, bt = _bufs(n), _bufs(n)
    nxt = _eventful_actions(n, 2)
    static_a = torch.zeros(n, 4, device=DEV)
    out = torch.zeros(16, dtype=torch.float64, device=DEV)
    a = nxt()
    static_a.copy_(a.to(DEV))
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        sim.step(static_a, *_args(b))             # one eager step on the capture stream before the capture
        with torch.cuda.graph(graph, stream=s):
            for _ in range(j):
                sim.step(static_a, *_args(b))
            sim.metrics(clear=True, out=out)
    torch.cuda.current_stream().wait_stream(s)
    twin.step(a.to(DEV), *_args(bt))
    ora.step(a)
    reads = [sim.metrics(clear=True).cpu().numpy()]
    for r in range(replays):
        a = nxt()
        static_a.copy_(a.to(DEV))
        graph.replay()
        reads.append(out.cpu().numpy().copy())
        for _ in range(j):
            twin.step(a.to(DEV), *_args(bt))
            ora.step(a)
    _in_step(b["reset"], b["progress"], ora, "graph")
    total, whole = np.sum(reads, axis=0), twin.metrics().cpu().numpy()
    assert np.array_equal(total[2:], whole[2:])
    assert_metrics(total, ora, "sum of captured clearing reads")
    assert_metrics(whole, ora, "eager twin")
    assert sim.step_count == 1 + j * replays and min(ora.counts[EPISODES], ora.counts[CRASH_Z], ora.counts[FAULT_STEPS]) > 0


@pytest.mark.parametrize("path", ["generic", "tma", "rollout"])
def test_collect_metrics_off_leaves_the_vector_zero_and_the_step_unchanged(path):
    n = 1001
    on, _ = _sim(n, tma=path == "tma", seed=6, **EVENTFUL)
    off, _ = _sim(n, tma=path == "tma", seed=6, collect_metrics=0, **EVENTFUL)
    bo, bf = _bufs(n), _bufs(n)
    nxt = _eventful_actions(n, 3)
    for t in range(20):
        if path == "rollout":
            on.rollout(3, bo["obs"], bo["rew"], bo["reset"], bo["progress"])
            off.rollout(3, bf["obs"], bf["rew"], bf["reset"], bf["progress"])
        else:
            a = nxt().to(DEV)
            on.step(a, *_args(bo))
            off.step(a, *_args(bf))
        for k in bo:
            assert torch.equal(bo[k], bf[k]), f"{path} t={t}: {k} differs with metrics off"
    so, sf = on.get_state(), off.get_state()
    for k in so:
        assert torch.equal(so[k], sf[k]), k
    po, pf = on.get_params(), off.get_params()
    assert torch.equal(po[0], pf[0]) and torch.equal(po[1], pf[1])
    assert on.step_count == off.step_count
    assert not off.metrics().cpu().numpy().any(), "collect_metrics=0 but the vector is not zero"
    mo = on.metrics().cpu().numpy()
    assert mo[8] == n * (60 if path == "rollout" else 20) and mo[9] > 0
