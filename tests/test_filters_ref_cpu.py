"""The exact CPU twin of the estimators (tests/filters_ref.c), checked without a GPU.

  * its float64 build restates the reference's algebra: it agrees with oracle/pv_filter.py and oracle/ahrs_ekf.py run in float64
    (the factored prediction, the rotated velocity block, the reused bias column and the cancelled bias terms included);
  * its float32 build, which the GPU tests hold the kernels to bit for bit, is as accurate as the reference's own float32 code on
    the reference's fixture, with the float64 build as arbiter.
"""
import os

import numpy as np
import pytest

import filters_ref as fr

G = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return np.load(os.path.join(G, name), allow_pickle=False)


def _spd_inputs(rng, n):
    """Well-conditioned random SPD covariances (max |P| <= 4, eigenvalues >= 0.1) and quaternions of norm 1e-3 .. 1e3."""
    A = rng.normal(size=(n, 9, 9))
    P = A @ np.swapaxes(A, 1, 2) / 9.0 + 0.1 * np.eye(9)
    P *= (rng.uniform(0.3, 1.0, size=n) * 4.0 / np.abs(P).max(axis=(1, 2)))[:, None, None]
    q = rng.normal(size=(n, 4))
    q *= (10.0 ** rng.uniform(-3, 3, size=n) / np.linalg.norm(q, axis=1))[:, None]
    return P.astype(np.float32), q.astype(np.float32)


def _rel_err(a, b, axes):
    return np.abs(a - b).max(axis=axes) / np.maximum(np.abs(b).max(axis=axes), 1e-300)


@pytest.mark.parametrize("flip_qw", [True, False])
@pytest.mark.parametrize("stages", ["predict", "pos", "vel", "predict+pos+vel"])
def test_float64_twin_restates_the_reference_algebra(stages, flip_qw):
    """float64 twin vs oracle/pv_filter.py in float64: <= 1e-12 relative per env, over four chained steps, R >= 1e-2 |P|."""
    from oracle.pv_filter import PVFilterBank
    n, f = 512, np.float64
    rng = np.random.default_rng(11 + 2 * len(stages) + int(flip_qw))
    P0, _ = _spd_inputs(rng, n)
    ora = PVFilterBank(n, [0.7, 1.3, 0.4], dtype=f)
    twin = fr.PVTwinBank(n, [0.7, 1.3, 0.4], dtype=f)
    x0 = rng.normal(size=(n, 9)).astype(np.float32)
    ora.state, ora.cov = x0.astype(f), P0.astype(f)
    twin.state, twin.cov = x0.astype(f), P0.astype(f)
    pos_var, vel_var = np.array([0.05, 0.08, 0.1]), np.array([0.1, 0.06, 0.04])
    for t in range(4):
        _, q = _spd_inputs(rng, n)
        acc = (rng.normal(size=(n, 3)) * 3).astype(np.float32)
        pm, vm = rng.normal(size=(n, 3)).astype(np.float32), rng.normal(size=(n, 3)).astype(np.float32)
        mask = rng.random(n) < 0.7
        if "predict" in stages:
            ora.prediction_step(acc, q, 0.02, flip_Qw=flip_qw)
            twin.prediction_step(acc, q, 0.02, flip_Qw=flip_qw)
        if "pos" in stages:
            for b in (ora, twin):
                b.correction_step(gps_data=pm, gps_var=pos_var, mask=mask)
        if "vel" in stages:
            for b in (ora, twin):                                   # gps_var given: the velocity fix uses vel_var
                b.correction_step(vel_data=vm, vel_var=vel_var, gps_var=pos_var, mask=mask)
        ex, eP = _rel_err(twin.state, ora.state, 1), _rel_err(twin.cov, ora.cov, (1, 2))
        assert ex.max() <= 1e-12 and eP.max() <= 1e-12, (t, ex.max(), eP.max())
        assert np.isfinite(twin.cov).all()


def test_ekf_twin_vs_oracle_fixture_and_known_answer():
    """The EKF twin (float64, the kernel's own normalisation and Gauss-Jordan inverse) against oracle/ahrs_ekf.py on the
    reference's fixture, fed the float32-rounded sensors the kernel takes; and SURVEY KAT-E."""
    from oracle.ahrs_ekf import EKFBank
    d = load("ekf.npz")
    T, n = d["gyr"].shape[:2]
    ora = EKFBank(n, 100.0)
    q_ora = d["q0"].copy()
    q4, P16 = d["q0"].T.copy(), np.eye(4).reshape(16, 1).repeat(n, 1)
    for t in range(T):
        g32, a32 = d["gyr"][t].astype(np.float32), d["ang"][t].astype(np.float32)
        q_ora = ora.update(q_ora / np.linalg.norm(q_ora, axis=1, keepdims=True), g32.astype(np.float64), a32.astype(np.float64))
        q4, P16 = fr.ekf_update(q4, P16, g32, a32, Dt=0.01)
        np.testing.assert_allclose(q4.T, q_ora, rtol=1e-9, atol=1e-12, err_msg=f"t={t}")
        np.testing.assert_allclose(P16.T.reshape(n, 4, 4), ora.P, rtol=1e-7, atol=1e-15, err_msg=f"t={t}")
        np.testing.assert_allclose(q4.T, d["Q"][t], rtol=0, atol=2e-7)
    # SURVEY KAT-E, with the xyzw input order and the float32 output the fused kernel uses (the fixture's kat_q was made from
    # float64 sensors: the float32 ones move it by ~1e-9)
    g, a = np.float32([[0.1, -0.2, 0.3]]), np.float32([[0.9990, 0.03, -0.02, 0.025]])
    q4, P16, q32 = fr.ekf_update(np.array([[1.0], [0], [0], [0]]), np.eye(4).reshape(16, 1), g, a[:, [1, 2, 3, 0]],
                                 ang_xyzw=True, q_f32_out=True)
    kq = EKFBank(1).update(np.array([[1.0, 0, 0, 0]]), g.astype(np.float64), a.astype(np.float64))
    np.testing.assert_allclose(q4[:, 0], kq[0], rtol=1e-9)
    np.testing.assert_allclose(q4[:, 0], d["kat_q"], rtol=1e-7)
    np.testing.assert_allclose(q4[:, 0], [0.99903697, 0.03000111, -0.02000074, 0.02500092], atol=1e-7)
    assert np.array_equal(q32[0], q4[:, 0].astype(np.float32))


def test_pv_twin_known_answer():
    """SURVEY KAT-V through the float32 twin: one prediction from rest, then a position fix."""
    d = load("pvfilter.npz")
    x, P = np.zeros((9, 1), np.float32), (np.eye(9, dtype=np.float32) * 1000).reshape(81, 1)
    x, P = fr.pv_step(x, P, accel=[[0, 0, 9.8]], quat=[[0, 0, 0, 1.0]], dt=0.01)
    np.testing.assert_allclose(x[:, 0], d["kat_pred"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(x[:, 0], [0, 0, 4.9e-4, 0, 0, 0.098, 0, 0, 0], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(np.diag(P.reshape(9, 9)), np.diag(d["kat_pred_cov"]), rtol=1e-6)
    x, P = fr.pv_step(x, P, pos_meas=[[1.0, 2.0, 3.0]], pos_var=[1e-7] * 3)
    np.testing.assert_allclose(x[:, 0], d["kat_corr"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(x[:3, 0], [1, 2, 3], atol=1e-5)


def test_float32_twin_is_as_accurate_as_the_reference():
    """DESIGN.md V2 bound, now on any machine: from the reference's own previous state (tests/golden/pvfilter.npz), the float32
    twin's error against the float64 twin is at most 4x the reference's own float32 error plus 8 float32 ulp of the scale, for
    the state and the covariance.  The kernels equal the float32 twin bit for bit (tests/test_gpu_filters_exact.py)."""
    from test_oracle_golden import pv_fixture_steps
    d = load("pvfilter.npz")
    floor = 8 * float(np.finfo(np.float32).eps)
    fixes = 0
    for t, ps, pc in pv_fixture_steps(d):
        n = ps.shape[0]
        kw = dict(accel=d["acc"][t], quat=d["quat"][t], pos_meas=d["pos_meas"][t], vel_meas=d["vel_meas"][t],
                  pos_mask=d["pos_fix"][t], vel_mask=d["vel_fix"][t], dt=0.01, flip_qw=(t % 2 == 0), pos_var=[1e-7] * 3)
        x32, P32 = fr.pv_step(ps.T, pc.reshape(n, 81).T, dtype=np.float32, **kw)        # velocity fix with R = 0, as the task
        x64, P64 = fr.pv_step(ps.T, pc.reshape(n, 81).T, dtype=np.float64, **kw)
        sref, cref = d["states"][t].T, d["covs"][t].reshape(n, 81).T
        sc, scc = np.abs(x64).max() + 1.0, np.abs(P64).max()
        e_ref_s, e_twin_s = np.abs(sref - x64).max() / sc, np.abs(x32 - x64).max() / sc
        e_ref_c, e_twin_c = np.abs(cref - P64).max() / scc, np.abs(P32 - P64).max() / scc
        assert e_twin_s <= 4.0 * e_ref_s + floor, (t, e_twin_s, e_ref_s)
        assert e_twin_c <= 4.0 * e_ref_c + floor, (t, e_twin_c, e_ref_c)
        fixes += int(d["pos_fix"][t].sum() + d["vel_fix"][t].sum())
    assert fixes > 0


def test_trigger_sweep_reaches_every_worker_count():
    """The trigger sweep of tests/test_gpu_filters_exact.py drives the cooperative fixes of the fused kernel through every worker
    count S = 1 .. 9 in both passes, the ragged last warp included (S = 7 needs one); checked from the trigger rule alone."""
    from test_gpu_filters_exact import SWEEP, SWEEP_STEPS
    u1, u2 = set(), set()
    for n, trig, per_env, base, total, s1, s2 in SWEEP:
        r1, r2 = fr.coop_worker_counts(n, SWEEP_STEPS, trig, per_env=per_env, env_id_base=base, n_total=total)
        assert s1 <= r1 and s2 <= r2, (n, trig, r1, r2)
        u1, u2 = u1 | s1, u2 | s2
    assert u1 == u2 == set(range(1, 10)), (u1, u2)
    # S = 7 is out of reach of full warps (32 lanes / 4 jobs = 8, / 5 jobs = 6): it comes from a ragged last warp
    assert fr.coop_worker_counts(992, SWEEP_STEPS, (8, 0, 8, 0)) == ({8}, {8})
