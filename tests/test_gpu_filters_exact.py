"""Every kernel that runs the estimators of ouzelum_b200/csrc/filters.cuh, bit for bit against the exact CPU twin tests/filters_ref.c.

The filters use only correctly rounded operations with explicit fused multiply-adds (every TU is built with -fmad=false), so the
float32 twin must reproduce every bit: comparisons are on the raw bits (signed zeros count), every compared value must be finite,
and multi-step sequences of the stand-alone banks run WITHOUT re-synchronising the twin from the device.
  * pv_step_kernel (PVFilterBank) and ekf_update_kernel (EKFBank) at 1 .. 2^20 + 3 envs
  * ekf_lee_fused_kernel, both instantiations (ozl_ekf_lee_step, ozl_ekf_lee_landed_step), at every launch shape it has (no tensor
    map, tensor-map box with zero-filled columns, plain-load fallback, ragged last warp, several waves), and a trigger sweep that
    drives the warp-cooperative fixes (pv_correct_coop) through every worker count S = 1 .. 9 in both passes
The Lee controller after the warm-up (libdevice atan2f / asinf / sincosf / fmodf) keeps the tolerance of test_gpu_config3.py.
"""
import numpy as np
import pytest
import torch

import filters_ref as fr

DEV = "cuda:0"
SIZES = [1, 127, 128, 129, 4099, 2 ** 20 + 3]


def assert_bits(dev, ref, what):
    """Raw-bit equality of a device array and its twin (same dtype and shape), both finite."""
    a = dev.detach().cpu().numpy() if torch.is_tensor(dev) else np.asarray(dev)
    b = np.asarray(ref)
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    assert np.isfinite(b).all(), f"{what}: twin produced non-finite values"
    assert np.isfinite(a).all(), f"{what}: kernel produced {int((~np.isfinite(a)).sum())} non-finite values"
    it = np.int32 if a.dtype.itemsize == 4 else np.int64
    diff = a.view(it) != b.view(it)
    if diff.any():
        idx = np.argwhere(diff)
        i0 = tuple(idx[0])
        raise AssertionError(f"{what}: {len(idx)} of {a.size} values differ in their bits; first at {i0}: kernel {a[i0]!r} "
                             f"twin {b[i0]!r}, max |diff| {np.abs(a.astype(np.float64) - b.astype(np.float64)).max():.3e}")


def _quats(rng, n):
    q = rng.normal(size=(n, 4))
    return (q * (10.0 ** rng.uniform(-3, 3, size=n) / np.linalg.norm(q, axis=1))[:, None]).astype(np.float32)


# ------------------------------------------------------------------------------------------------ K3 stand-alone
@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["task", "well_conditioned"])
@pytest.mark.parametrize("n", SIZES)
def test_pv_step_kernel_equals_twin(n, regime):
    """`ozl_pv_step` over a sequence of steps, the twin running alongside on its own state.  task: P = 1000 I collapsing to
    ~1e-7 under position fixes with R = 1e-7 and velocity fixes with R = 0; well_conditioned: SPD P of order 1, R >= 1e-2 |P|.
    Covers predict on / off, both flip_qw, per-env masks and the period rule with a non-zero iter_base, |q| from 1e-3 to 1e3."""
    from ouzelum_b200.pv_filter import PVFilterBank
    rng = np.random.default_rng(n + (0 if regime == "task" else 7))
    steps = 6 if n > 100000 else 40
    task = regime == "task"
    acc_var = [1.0, 1.0, 1.0] if task else [0.7, 1.3, 0.4]
    bank = PVFilterBank(n, acc_var, DEV)
    if task:
        x, P = np.zeros((9, n), np.float32), np.repeat((np.eye(9, dtype=np.float32) * 1000).reshape(81, 1), n, 1)
        pos_var, vel_var, dt = [1e-7] * 3, None, 0.01
    else:
        A = rng.normal(size=(n, 9, 9)).astype(np.float32)
        P = (A @ np.swapaxes(A, 1, 2) / np.float32(9) + np.float32(0.1) * np.eye(9, dtype=np.float32)).reshape(n, 81).T.copy()
        x = rng.normal(size=(9, n)).astype(np.float32)
        pos_var, vel_var, dt = [0.3, 0.5, 0.4], [0.2, 0.6, 0.3], 0.02
    bank.set_states(torch.from_numpy(x.T.copy()))
    bank.set_covariances(torch.from_numpy(P.T.copy()))
    t_ = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    fixes = 0
    for t in range(steps):
        predict = t % 5 != 4
        acc = (rng.normal(size=(n, 3)) * 3).astype(np.float32) if predict else None
        q = _quats(rng, n) if predict else None
        pm = (rng.normal(size=(n, 3)) * 5).astype(np.float32)
        # no velocity fix without a prediction in the task regime: two R = 0 fixes back to back leave S singular
        vm = rng.normal(size=(n, 3)).astype(np.float32) if (predict or not task) else None
        pmask = vmask = trig = None
        iter_base = 0
        if t % 3 == 0:
            pmask, vmask = rng.random(n) < 0.3, rng.random(n) < 0.35
        elif t % 3 == 1:
            trig, iter_base = (7, 6, 3, 0), t * n + 12345
        else:
            trig, iter_base = (2, 1, 5, 3), 2 ** 33 + 3 * t
        bank.step(accels=t_(acc), orientation=t_(q), dt=dt, flip_Qw=(t % 2 == 0), gps_data=t_(pm), gps_var=pos_var,
                  gps_mask=t_(pmask), vel_data=t_(vm), vel_var=vel_var, vel_mask=t_(vmask), trigger=trig, iter_base=iter_base)
        x, P = fr.pv_step(x, P, accel=acc, quat=q, pos_meas=pm, vel_meas=vm, pos_mask=pmask, vel_mask=vmask, dt=dt,
                          acc_var=acc_var, pos_var=pos_var, vel_var=vel_var, flip_qw=(t % 2 == 0), trigger=trig, iter_base=iter_base)
        assert_bits(bank._x, x, f"PV x t={t}")
        assert_bits(bank._P, P, f"PV P t={t}")
        pos_fixed = pmask if pmask is not None else (iter_base + np.arange(n)) % trig[0] == trig[1]
        fixes += int(pos_fixed.sum())
    assert fixes > 0
    if task and (n > 1 or pos_fixed.any()):
        # the task regime reached: a position fix with R = 1e-7 brings the position variances from up to ~1e3 down to the order
        # of R (the R = 0 velocity fix after it only lowers them); float32 cancellation in (I - KH) P leaves a residue of a few
        # ulp of the prior, up to ~2e-3 where the prior was never fixed before.  Envs not fixed in the last step keep growing.
        assert pos_fixed.any()
        v = np.abs(P[[0, 10, 20]][:, pos_fixed])
        assert np.median(v) < 1e-6 and v.max() < 1e-2, (np.median(v), v.max())


# ------------------------------------------------------------------------------------------------ K2 stand-alone
@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_ekf_update_kernel_equals_twin(n):
    """`ozl_ekf_update` over a sequence of steps from unnormalised quaternions: q and P (float64) and the float32 copy of q, with
    the measurement in both orders (wxyz, xyzw)."""
    from ouzelum_b200.ahrs_ekf import EKFBank
    rng = np.random.default_rng(100 + n)
    steps = 4 if n > 100000 else 20
    bank = EKFBank(n, frequency=100.0, device=DEV)
    q0 = _quats(rng, n).astype(np.float64)
    bank.set_state(torch.from_numpy(q0))
    q4, P16 = q0.T.copy(), np.repeat(np.eye(4).reshape(16, 1), n, 1)
    for t in range(steps):
        gyr = (rng.normal(size=(n, 3)) * 2).astype(np.float32)
        ang = (q4.T + rng.normal(size=(n, 4)) * 0.05).astype(np.float32)
        xyzw = t % 2 == 1
        if xyzw:
            ang = ang[:, [1, 2, 3, 0]].copy()
        q32 = torch.zeros(n, 4, device=DEV) if t % 3 != 2 else None
        bank.update(torch.from_numpy(gyr), torch.from_numpy(ang), ang_xyzw=xyzw, q_f32_out=q32)
        out = fr.ekf_update(q4, P16, gyr, ang, ang_xyzw=xyzw, Dt=bank.Dt, g_noise=bank.g_noise, q_f32_out=q32 is not None)
        q4, P16 = out[0], out[1]
        assert_bits(bank._q, q4, f"EKF q t={t}")
        assert_bits(bank._P, P16, f"EKF P t={t}")
        if q32 is not None:
            assert_bits(q32, out[2], f"EKF q float32 t={t}")


# ------------------------------------------------------------------------------------------------ fused estimator step
def _twin_glue(env, n, **kw):
    from oracle.ekf_lee_landed import EKFLeeGlue

    class TwinGlue(EKFLeeGlue):
        """The glue of EKFLeeLanded with the exact twin in place of the reference-algebra filter oracles."""

        def __init__(self):
            super().__init__(n, **kw)
            self.ekf = fr.EKFTwinBank(self, n, Dt=self.ekf.Dt, g_noise=self.ekf.g_noise)
            self.pv = fr.PVTwinBank(n, [1.0, 1.0, 1.0])

    g = TwinGlue()
    assert g.ekf.Dt == env._fa.ekf_Dt and g.ekf.g_noise == env._fa.ekf_g_noise
    return g


def run_fused_vs_twin(n, fused_step=True, trigger=None, per_env=False, env_id_base=0, n_total=None, steps=7, conv=3, seed=21):
    """Snapshot pattern of test_gpu_config3.py: the device state is copied into the twin glue before every step, the kernel and
    the glue then advance once, and every estimator output is compared bit for bit.  Returns (resets seen, sensor fixes)."""
    import ouzelum_b200
    from oracle.lee_control import lee_control
    from oracle.quad_step import QuadStepOracle
    from test_gpu_config3 import _snapshot_into
    extra = {}
    if env_id_base or n_total:
        extra = dict(envIdBase=env_id_base, numEnvsTotal=n_total)
    cfg = ouzelum_b200.task_config("EKFLeeLanded", n, seed=seed, POMDP="flickering_and_random_noise", pomdp_prob=0.1,
                                   ConvergenceTime=conv, maxEpisodeLength=5, exposeEstimates=True, fusedStep=fused_step,
                                   perEnvSensorTriggers=per_env, **extra)
    env = ouzelum_b200.make(seed=seed, task="EKFLeeLanded", num_envs=n, sim_device=DEV, rl_device=DEV, headless=True, cfg=cfg)
    assert env.fused and env.fused_step == fused_step
    if trigger is not None:
        env._fa.pos_period, env._fa.pos_phase, env._fa.vel_period, env._fa.vel_phase = trigger
    trig = (env._fa.pos_period, env._fa.pos_phase, env._fa.vel_period, env._fa.vel_phase)
    phys = QuadStepOracle(env.native_cfg.to_dict())
    glue = _twin_glue(env, n, convergence=conv, pomdp_mode=3, pomdp_prob=0.1, seed=seed, env_id_base=env_id_base, trigger=trig,
                      per_env_triggers=per_env, n_total=n_total)
    a = torch.zeros(n, 4, device=DEV)
    n_reset = n_fix = 0
    for t in range(steps):
        _snapshot_into(env, phys, glue, t)
        reset_before = env.reset_buf.bool().cpu().numpy().copy()
        n_reset += int(reset_before.sum())
        env.step(a)
        tgt = env.husky.target.cpu().numpy()
        root = phys.post_reset_root().numpy()
        wrench_o, est_o, cmd_o = glue.pre_physics(root, tgt, reset_before)
        assert_bits(env.ekf._q, np.ascontiguousarray(glue.Q.T), f"EKF q t={t}")
        assert_bits(env.ekf._P, np.ascontiguousarray(glue.ekf.P.reshape(n, 16).T), f"EKF P t={t}")
        assert_bits(env.pvfilters._x, np.ascontiguousarray(glue.pv.state.T), f"PV x t={t}")
        assert_bits(env.pvfilters._P, np.ascontiguousarray(glue.pv.cov.reshape(n, 81).T), f"PV P t={t}")
        assert_bits(env.prev_root_linvels, glue.prev_v, f"prev_root_linvels t={t}")
        assert_bits(env.target_waypoints, glue.waypoints, f"target_waypoints t={t}")
        assert_bits(env._cmd, cmd_o, f"cmd t={t}")
        assert_bits(env._est, est_o, f"est t={t}")
        w = env._wrench.cpu().numpy()
        if t < conv:
            assert_bits(w, wrench_o, f"hover wrench t={t}")
        else:
            # Lee (libdevice transcendentals): compared on the kernel's own, bit-checked estimate at test_gpu_config3's tolerance
            th, tq = lee_control(env._est.cpu().numpy(), env._cmd.cpu().numpy(), mode=0)
            np.testing.assert_allclose(w[:, 0], glue.mg * th, rtol=2e-5, atol=2e-4, err_msg=f"thrust t={t}")
            np.testing.assert_allclose(w[:, 1:], tq, rtol=2e-5, atol=1e-4, err_msg=f"torque t={t}")
        ids = np.arange(n, dtype=np.int64) + env_id_base
        k = np.full(n, t) if per_env else t * int(n_total or n) + ids
        n_fix += int(((k % trig[0]) == trig[1]).sum() + ((k % trig[2]) == trig[3]).sum())
    assert steps > conv
    return n_reset, n_fix


# n < 32: no tensor map; 36, 100, 4100: tensor-map box with zero-filled columns past N and a partial last CTA; 95, 961, 4099:
# n % 4 != 0, plain-load fallback and a ragged last warp; 65536: config 3; 100000: more than one wave of 96-env CTAs (eager)
FUSED_SHAPES = [1, 31, 36, 100, 4100, 95, 961, 4099]


@pytest.mark.gpu
@pytest.mark.parametrize("fused_step", [True, False], ids=["landed_step", "ekf_lee_step"])
@pytest.mark.parametrize("n", FUSED_SHAPES + [65536, 100000])
def test_fused_estimator_step_equals_twin(n, fused_step):
    if n > 4100 and not fused_step:
        pytest.skip("the large shapes run on the default one-launch step only")
    n_reset, n_fix = run_fused_vs_twin(n, fused_step=fused_step)
    assert n_reset > n and n_fix > 0


# (n, trigger, per-env triggers, envIdBase, numEnvsTotal, worker counts claimed in pass 1, in pass 2); 7 steps each
SWEEP = [
    (999, (8, 0, 8, 0), False, 0, None, {7, 8}, {7, 8}),
    (1020, (11, 4, 16, 9), False, 0, None, {5, 6, 7, 8, 9}, {9}),
    (961, (5, 0, 5, 0), False, 0, None, {1, 4, 5}, {1, 4, 5}),
    (961, (6, 0, 6, 0), False, 0, None, {1, 5, 6}, {1, 5, 6}),
    (961, (2, 0, 2, 0), False, 0, None, {1, 2}, {1, 2}),
    (4099, (3, 2, 4, 1), False, 0, None, {1, 2, 3}, {3, 9}),
    (961, (33, 7, 1, 0), False, 0, None, {1}, {1, 9}),
    (999, (4, 1, 4, 1), False, 0, None, {3, 4, 7}, {3, 4, 7}),
    (999, (7, 6, 3, 0), True, 0, None, {1}, {1}),                   # perEnvSensorTriggers: all lanes fix together
    (1000, (7, 6, 3, 0), False, 3000, 8000, {2, 4}, {8, 9}),        # one shard of a larger job
]
SWEEP_STEPS = 7


@pytest.mark.gpu
@pytest.mark.parametrize("n,trigger,per_env,base,total,s1,s2", SWEEP)
def test_fused_cooperative_fixes_equal_twin_at_every_worker_count(n, trigger, per_env, base, total, s1, s2):
    r1, r2 = fr.coop_worker_counts(n, SWEEP_STEPS, trigger, per_env=per_env, env_id_base=base, n_total=total)
    assert s1 <= r1 and s2 <= r2, (r1, r2)
    run_fused_vs_twin(n, trigger=trigger, per_env=per_env, env_id_base=base, n_total=total, steps=SWEEP_STEPS)
