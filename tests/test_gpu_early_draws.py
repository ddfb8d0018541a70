"""Sub-wave step kernel (quad_step_subwave_kernel: launches of up to 4 x 128-env CTAs per SM; override OZL_EARLY_DRAW_MAX_ENVS,
read once per handle at ozl_create).  It draws the reset-path Philox numbers of every env ahead of the state's first use; every
output must stay bit-identical to the default kernel's, on every task whose step launches can select it, with and without a
states output and a scenario table, over enough steps for resets and target re-samples to occur."""
import os

import pytest
import torch

import scenario_ref as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
VAR = "OZL_EARLY_DRAW_MAX_ENVS"
STEPS = 300


def _task(name, n, early, states=False, scn=False):
    """early: True = the sub-wave kernel at any size, False = never, None = the library's default selection."""
    import ouzelum_b200
    extra = dict(maxEpisodeLength=40, asymmetric_observations=states)
    if name != "LeeLanded":                       # LeeLanded is wrench-actuated: no rotor faults
        extra.update(rotorFault={"enable": True})
    if name == "Ouzelum":
        extra.update(domainRandomization={"enable": True})
    old = os.environ.get(VAR)
    if early is not None:
        os.environ[VAR] = str(1 << 40) if early else "0"
    else:
        os.environ.pop(VAR, None)
    try:
        env = ouzelum_b200.make(seed=21, task=name, num_envs=n, sim_device=DEV, rl_device=DEV, headless=True,
                                cfg=ouzelum_b200.task_config(name, n, seed=21, **extra))
    finally:
        if old is None:
            os.environ.pop(VAR, None)
        else:
            os.environ[VAR] = old
    if scn:
        env.set_scenarios(S.mixed_rows(n, env.native_cfg.to_dict(), seed=4))
    return env


def _outputs(env, states):
    st = env.sim.get_state()
    params, fault = env.sim.get_params()
    out = dict(obs=env.obs_buf, rew=env.rew_buf, reset=env.reset_buf, progress=env.progress_buf, timeout=env.timeout_buf,
               ep_ret=env.episode_return_buf, params=params, fault=fault, metrics=env.metrics(),
               **{"st_" + k: v for k, v in st.items()})
    if states:
        out["states"] = env.states_buf
    return {k: v.clone() for k, v in out.items()}


def _bits(t):
    """Raw bits of a float tensor (signed zeros and NaN payloads count), the tensor itself otherwise."""
    return t.view({torch.float32: torch.int32, torch.float64: torch.int64}[t.dtype]) if t.is_floating_point() else t


def _assert_bit_equal(x, y, what):
    for k in y:
        assert torch.equal(_bits(x[k]), _bits(y[k])), f"{what}: {k}"


def _run_pair(name, n, states, scn, a_early, b_early, steps=STEPS):
    a, b = _task(name, n, a_early, states, scn), _task(name, n, b_early, states, scn)
    g = torch.Generator().manual_seed(3)
    for t in range(steps):
        act = ((torch.rand(n, 4, generator=g) * 2 - 1) * 0.6).to(DEV)
        a.step(act)
        b.step(act)
        if t % 25 == 24 or t == steps - 1:
            _assert_bit_equal(_outputs(a, states), _outputs(b, states), f"{name} n={n} t={t}")
    return b.metrics().cpu()


@pytest.mark.parametrize("n", [37, 4099, 16384])
@pytest.mark.parametrize("name", ["Ouzelum", "Landing", "Landed", "LeeLanded"])
@pytest.mark.parametrize("states,scn", [(False, False), (True, False), (False, True), (True, True)])
def test_subwave_kernel_equals_default_kernel(name, n, states, scn):
    m = _run_pair(name, n, states, scn, True, False)
    assert m[9] > 0 and m[15] > 0, m                  # episodes ended and resets were applied: the early draws were used
    if name != "LeeLanded":
        assert m[14] > 0, m                           # rotor faults were active


def _kernel_names(env, n):
    from torch.profiler import ProfilerActivity, profile
    act = torch.zeros(n, 4, device=DEV)
    env.step(act)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        env.step(act)
        torch.cuda.synchronize()
    return " ".join(e.name for e in prof.events())


@pytest.mark.parametrize("side", ["below", "above"])
def test_default_selection_at_the_threshold(side):
    """One wave of the sub-wave kernel (4 x 128-env CTAs per SM) is the default limit: the default handle runs the kernel the
    forced one does, with the same bits."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    limit = 4 * 128 * sms
    n = limit if side == "below" else limit + 1
    early = side == "below"
    names = _kernel_names(_task("Ouzelum", n, None), n)
    assert ("quad_step_subwave_kernel" in names) == early, names
    assert ("quad_step_kernel" in names) == (not early), names
    m = _run_pair("Ouzelum", n, False, False, None, early, steps=120)
    assert m[9] > 0, m
