#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ by RUNNING THE REFERENCE'S OWN CODE (CPU, this container only).

    python tests/golden/make_golden.py [/root/reference]

The reference package cannot be imported whole (isaacgym / gym / hydra / ahrs are absent), so
  * `isaacgymenvs` is registered as a bare namespace package pointing at the checkout, which makes
    `isaacgymenvs.controllers.*`, `isaacgymenvs.PVFilter`, `isaacgymenvs.utils.trajectories`,
    `isaacgymenvs.utils.controllers` importable unmodified;
  * the `@torch.jit.script` reward functions and `quat_axis` / `my_quat_rotate` are lifted out of their
    modules with `ast` (their modules import isaacgym at the top) and exec'd as plain Python;
  * `isaacgymenvs.ahrs_ekf` is imported with a stub `ahrs` package that supplies only `skew` (the one
    third-party helper on the executed branch), `q2R/ecompass/acc2q/cosd/sind` placeholders and a dummy WMM.
Nothing in tests/, bench.py or smoke() reads the reference at run time: they read the .npz files written here.
"""
import ast
import os
import sys
import types

import numpy as np
import torch

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REF, "isaacgymenvs")


def install_namespace():
    m = types.ModuleType("isaacgymenvs")
    m.__path__ = [PKG]
    sys.modules["isaacgymenvs"] = m


def lift(path, names, extra_globals=None):
    """exec the named top-level functions of `path` (decorators stripped) and return them."""
    src = open(path).read()
    tree = ast.parse(src)
    g = {"torch": torch, "Tensor": torch.Tensor, "Tuple": tuple}
    g.update(extra_globals or {})
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            node.decorator_list = []
            code = compile(ast.Module(body=[node], type_ignores=[]), path, "exec")
            exec(code, g)
    return [g[n] for n in names]


def stub_ahrs():
    def skew(x):
        return np.array([[0.0, -x[2], x[1]], [x[2], 0.0, -x[0]], [-x[1], x[0], 0.0]])

    ahrs = types.ModuleType("ahrs")
    common = types.ModuleType("ahrs.common")
    orientation = types.ModuleType("ahrs.common.orientation")
    mathfuncs = types.ModuleType("ahrs.common.mathfuncs")
    utils = types.ModuleType("ahrs.utils")
    wmm = types.ModuleType("ahrs.utils.wmm")
    for n in ("q2R", "ecompass", "acc2q"):
        setattr(orientation, n, lambda *a, **k: (_ for _ in ()).throw(NotImplementedError(n)))
    mathfuncs.cosd = lambda x: np.cos(np.radians(x))
    mathfuncs.sind = lambda x: np.sin(np.radians(x))
    mathfuncs.skew = skew
    mathfuncs.MUNICH_LATITUDE, mathfuncs.MUNICH_LONGITUDE, mathfuncs.MUNICH_HEIGHT = 48.1372, 11.5755, 0.519

    class WMM:                                    # result unused on the executed branch (SURVEY 8a row E1)
        def __init__(self, **kw):
            self.X, self.Y, self.Z = 21018.3, 1591.8, 43985.5
    wmm.WMM = WMM
    for name, mod in [("ahrs", ahrs), ("ahrs.common", common), ("ahrs.common.orientation", orientation),
                      ("ahrs.common.mathfuncs", mathfuncs), ("ahrs.utils", utils), ("ahrs.utils.wmm", wmm)]:
        sys.modules[name] = mod


def rand_states(n, g, spread=3.0):
    s = torch.zeros(n, 13)
    s[:, 0:3] = (torch.rand(n, 3, generator=g) * 2 - 1) * spread
    q = torch.randn(n, 4, generator=g)
    s[:, 3:7] = q / q.norm(dim=1, keepdim=True)
    s[:, 7:10] = torch.randn(n, 3, generator=g) * 2
    s[:, 10:13] = torch.randn(n, 3, generator=g) * 3
    return s


def main():
    install_namespace()
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(20261018)
    made = []

    # ---------------------------------------------------------------- reward / quat helpers (jit functions, lifted)
    tj = os.path.join(PKG, "utils", "torch_jit_utils.py")
    (my_quat_rotate,) = lift(tj, ["my_quat_rotate"])
    (quat_axis,) = lift(tj, ["quat_axis"], {"quat_rotate": my_quat_rotate})   # torch_jit_utils.py:198 == isaacgym quat_rotate
    helpers = {"quat_axis": quat_axis, "quat_rotate": my_quat_rotate}
    (rew_ouz,) = lift(os.path.join(PKG, "tasks", "ouzelum.py"), ["compute_ingenuity_reward"], helpers)
    (rew_land,) = lift(os.path.join(PKG, "tasks", "landing.py"), ["compute_ingenuity_reward"], helpers)
    (rew_quad,) = lift(os.path.join(PKG, "tasks", "quadcopter.py"), ["compute_quadcopter_reward"], helpers)
    n = 4096
    st = rand_states(n, g, spread=6.0)
    st[: n // 4, 3:7] = torch.tensor([0.0, 0.0, 0.0, 1.0]) + 0.05 * torch.randn(n // 4, 4, generator=g)   # near-upright, non-unit
    tgt = (torch.rand(n, 3, generator=g) * 2 - 1) * 5
    prog = torch.randint(0, 2100, (n,), generator=g)
    reset_in = torch.zeros(n, dtype=torch.long)
    r1, d1 = rew_ouz(st[:, 0:3], tgt, st[:, 3:7], st[:, 7:10], st[:, 10:13], reset_in, prog, 2000.0)
    r2, d2 = rew_land(st[:, 0:3], tgt, st[:, 3:7], st[:, 7:10], st[:, 10:13], torch.zeros(n, 6, 3), reset_in, prog, 2000.0)
    r3, d3 = rew_quad(st[:, 0:3], st[:, 3:7], st[:, 7:10], st[:, 10:13], reset_in, prog, 500.0)
    v = torch.randn(n, 3, generator=g)
    np.savez_compressed(os.path.join(OUT, "reward.npz"), state=st.numpy(), target=tgt.numpy(), progress=prog.numpy(),
                        rew_ouzelum=r1.numpy(), reset_ouzelum=d1.numpy(), rew_landing=r2.numpy(), reset_landing=d2.numpy(),
                        rew_quadcopter=r3.numpy(), reset_quadcopter=d3.numpy(),
                        quat_axis2=quat_axis(st[:, 3:7], 2).numpy(), rot_v=v.numpy(),
                        quat_rotate=my_quat_rotate(st[:, 3:7], v).numpy())
    made.append("reward.npz")

    # ---------------------------------------------------------------- Lee controllers (reference classes, unmodified)
    from isaacgymenvs.controllers.controller import Controller
    from isaacgymenvs.controllers.control_config import control
    n = 2048
    st = rand_states(n, g)
    st[:8, 3:7] = torch.tensor([0.0, 0.0, 0.0, 1.0])
    cmd = torch.zeros(n, 4)
    cmd[:, 0:3] = (torch.rand(n, 3, generator=g) * 2 - 1) * 3
    cmd[:, 3] = (torch.rand(n, generator=g) * 2 - 1) * 3.1
    out = {"state": st.numpy(), "command": cmd.numpy()}
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for name in ("lee_position_control", "lee_velocity_control", "lee_attitude_control"):
            cc = control()
            cc.controller = name
            c = Controller(cc, "cpu")
            thrust, torque = c(st.clone(), cmd.clone())
            out[name + "_thrust"] = thrust.numpy()
            out[name + "_torque"] = torque.numpy()
        # SURVEY 8c known answers
        c = Controller(control(), "cpu")
        s1 = torch.zeros(2, 13)
        s1[0, 2] = 1.0
        s1[0, 6] = 1.0
        s1[1, 3], s1[1, 6] = np.sin(0.1), np.cos(0.1)
        s1[1, 7:10] = torch.tensor([0.1, 0.0, -0.2])
        s1[1, 10:13] = torch.tensor([0.0, 0.1, 0.0])
        t1, q1 = c(s1, torch.tensor([[0.0, 0.0, 1.0, 0.0]] * 2))
        out["kat_state"], out["kat_thrust"], out["kat_torque"] = s1.numpy(), t1.numpy(), q1.numpy()
    np.savez_compressed(os.path.join(OUT, "lee.npz"), **out)
    made.append("lee.npz")

    # ---------------------------------------------------------------- PV filter (reference class, one object per env)
    from isaacgymenvs.PVFilter import PVFilter
    n, T = 24, 12
    acc_var = torch.tensor([1.0, 1.0, 1.0])
    filters = [PVFilter(acc_var, "cpu") for _ in range(n)]
    acc = torch.randn(T, n, 3, generator=g) * 2
    acc[..., 2] += 9.8
    quat = torch.randn(T, n, 4, generator=g)
    quat = quat / quat.norm(dim=-1, keepdim=True)
    pos_meas = torch.randn(T, n, 3, generator=g)
    vel_meas = torch.randn(T, n, 3, generator=g)
    var = torch.tensor([1.0, 1.0, 1.0]) * 0.0000001
    states = np.zeros((T, n, 9), np.float32)
    covs = np.zeros((T, n, 9, 9), np.float32)
    pos_fix = np.zeros((T, n), bool)
    vel_fix = np.zeros((T, n), bool)
    for t in range(T):
        for i, f_ in enumerate(filters):
            k = t * n + i                                       # global iteration index (SURVEY 8a row E3)
            f_.prediction_step(acc[t, i], quat[t, i], dt=0.01, sim_time=0.0, flip_Qw=(t % 2 == 0))
            if k % 7 == 6:
                f_.correction_step(gps_data=pos_meas[t, i], gps_var=var)
                pos_fix[t, i] = True
            if k % 3 == 0:
                f_.correction_step(vel_data=vel_meas[t, i], vel_var=var)       # gps_var=None => R = 0 (PVFilter.py:76-79)
                vel_fix[t, i] = True
            states[t, i] = f_.get_states().reshape(9).numpy()
            covs[t, i] = f_.get_covariances().numpy()
    # SURVEY KAT-V
    kf = PVFilter(acc_var, "cpu")
    kf.prediction_step(torch.tensor([0.0, 0.0, 9.8]), torch.tensor([0.0, 0.0, 0.0, 1.0]), dt=0.01)
    kat_pred = kf.get_states().reshape(9).numpy().copy()
    kat_pred_cov = kf.get_covariances().numpy().copy()
    kf.correction_step(gps_data=torch.tensor([1.0, 2.0, 3.0]), gps_var=var)
    np.savez_compressed(os.path.join(OUT, "pvfilter.npz"), acc=acc.numpy(), quat=quat.numpy(), pos_meas=pos_meas.numpy(),
                        vel_meas=vel_meas.numpy(), pos_fix=pos_fix, vel_fix=vel_fix, states=states, covs=covs,
                        kat_pred=kat_pred, kat_pred_cov=kat_pred_cov, kat_corr=kf.get_states().reshape(9).numpy(),
                        kat_corr_cov=kf.get_covariances().numpy())
    made.append("pvfilter.npz")

    # ---------------------------------------------------------------- trajectories + differential drive
    from isaacgymenvs.utils import trajectories as rt
    from isaacgymenvs.utils import controllers as rc
    n = 1024
    cur = (torch.rand(n, 2, generator=g) * 2 - 1) * 5
    tg = (torch.rand(n, 2, generator=g) * 2 - 1) * 5
    tg[:16] = cur[:16] + 0.001
    hd = torch.rand(n, generator=g) * 2 * np.pi                 # get_euler_xyz range [0, 2pi)
    dd = rc.differential_drive(cur, tg, hd.clone(), (3.0, 1000))
    dd_kat = rc.differential_drive(torch.zeros(2, 2), torch.tensor([[1.0, 0.0], [0.0, 1.0]]), torch.zeros(2), (3, 1000))
    np.savez_compressed(os.path.join(OUT, "trajectories.npz"), lemniscate=rt.lemniscate(a=4, num_points=100).numpy(),
                        circle=rt.circle(r=2, num_points=100).numpy(), square=rt.square(side_length=4, num_points=8).numpy(),
                        dd_cur=cur.numpy(), dd_tgt=tg.numpy(), dd_heading=hd.numpy(), dd_out=dd.numpy(), dd_kat=dd_kat.numpy())
    made.append("trajectories.npz")

    # ---------------------------------------------------------------- AHRS EKF (reference class, `ahrs` stubbed)
    stub_ahrs()
    from isaacgymenvs.ahrs_ekf import EKF
    n, T = 16, 20
    gn = np.random.default_rng(7)
    ekfs = [EKF(frequency=100.0) for _ in range(n)]
    q = gn.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q0 = q.copy()
    gyr = gn.normal(size=(T, n, 3)) * 2
    accs = gn.normal(size=(T, n, 3)) + np.array([0, 0, 9.8])
    ang = gn.normal(size=(T, n, 4)) * 0.05
    Q = np.zeros((T, n, 4))
    P = np.zeros((T, n, 4, 4))
    true_q = q.copy()
    for t in range(T):
        for i in range(n):
            meas = true_q[i] + ang[t, i]
            ang[t, i] = meas
            q[i] = ekfs[i].update(q=q[i] / np.linalg.norm(q[i]), gyr=gyr[t, i], acc=accs[t, i], ang=meas)
            Q[t, i], P[t, i] = q[i], ekfs[i].P
    e = EKF(frequency=100.0)
    kat_q = e.update(q=np.array([1.0, 0, 0, 0]), gyr=np.array([0.1, -0.2, 0.3]), acc=np.array([0.0, 0.0, 9.8]),
                     ang=np.array([0.9990, 0.03, -0.02, 0.025]))
    np.savez_compressed(os.path.join(OUT, "ekf.npz"), q0=q0, gyr=gyr, acc=accs, ang=ang, Q=Q, P=P, kat_q=kat_q, kat_P=e.P)
    made.append("ekf.npz")

    # ---------------------------------------------------------------- termination fixtures from the logged runs
    import glob
    rows = []
    for path in sorted(glob.glob(os.path.join(PKG, "trajectories", "flicker_0.01_ep_*.csv")),
                       key=lambda s: int(s.rsplit("_", 1)[1].split(".")[0])):
        ep = int(path.rsplit("_", 1)[1].split(".")[0])
        with open(path) as fh:
            has_header = fh.readline().startswith("Position")      # only ep_0 (opened in __init__, landed.py:114-117) has one
        with open(path) as fh:
            lines = fh.readlines()[1 if has_header else 0:]
        data = np.asarray([[float(x) for x in ln.split(",")] for ln in lines if ln.strip()], dtype=np.float64).reshape(-1, 6)
        if data.size == 0:
            rows.append((ep, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0))
            continue
        d = np.linalg.norm(data[:, 0:3] - data[:, 3:6], axis=1)
        prev_d = d[-2] if len(d) > 1 else np.nan
        rows.append((ep, len(data), d[-1], prev_d, data[-1, 2], data[:, 5].min(), data[:, 5].max(), d.min(),
                     data[0, 0], data[0, 1], data[0, 2]))
    counter = int(open(os.path.join(PKG, "metrics", "flicker_0.01.txt")).read().strip())
    np.savez_compressed(os.path.join(OUT, "landed_logs.npz"),
                        episodes=np.asarray(rows, dtype=np.float64),
                        columns=np.asarray(["episode", "rows", "last_dist", "prev_dist", "last_z", "target_z_min", "target_z_max",
                                            "min_dist", "x0", "y0", "z0"]),
                        landing_counter=counter)
    made.append("landed_logs.npz")

    # ---------------------------------------------------------------- RPO-LSTM Actor (config 5 / SURVEY 8f rank 1)
    # the reference's own module (RPO-LSTM/model.py:11-68), unmodified, on CPU: weights after ITS initialisation, a 3-step sequence
    # through get_states / forward (action=None: the collection path; the update path hard-codes "cuda:0", model.py:65)
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_rpo_lstm_model", os.path.join(PKG, "RPO-LSTM", "model.py"))
    ref_model = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_model)

    class _Space:
        def __init__(self, *shape):
            self.shape = shape
    torch.manual_seed(1234)
    actor = ref_model.Actor(_Space(13), _Space(4))
    with torch.no_grad():
        actor.actor_logstd.copy_(torch.tensor([[-0.3, 0.1, 0.0, 0.4]]))       # a trained-looking log-std, so that entropy / log-prob are not trivial
    B, T = 7, 3
    g = torch.Generator().manual_seed(5)
    obs = torch.randn(T * B, 13, generator=g)
    done = (torch.rand(T * B, generator=g) < 0.3).float()
    h0, c0 = torch.randn(1, B, 128, generator=g) * 0.5, torch.randn(1, B, 128, generator=g) * 0.5
    torch.manual_seed(99)
    with torch.no_grad():
        # one step (collection, main.py:95) and a T-step sequence (update path shapes, agent.py:95-100)
        a1, lp1, en1, (h1, c1) = actor(obs[:B], (h0, c0), done[:B])
        aT, lpT, enT, (hT, cT) = actor(obs, (h0, c0), done)
    sd = {"sd__" + k: v.numpy() for k, v in actor.state_dict().items()}
    np.savez_compressed(os.path.join(OUT, "rpo_lstm_actor.npz"), obs=obs.numpy(), done=done.numpy(), h0=h0.numpy(), c0=c0.numpy(),
                        a1=a1.numpy(), lp1=lp1.numpy(), en1=en1.numpy(), h1=h1.numpy(), c1=c1.numpy(),
                        aT=aT.numpy(), lpT=lpT.numpy(), enT=enT.numpy(), hT=hT.numpy(), cT=cT.numpy())
    # the state dict goes into two more files so that every stored file stays under 1 MB
    np.savez_compressed(os.path.join(OUT, "rpo_lstm_actor_sd_mlp.npz"), **{k: v for k, v in sd.items() if not k.startswith("sd__lstm.")})
    np.savez_compressed(os.path.join(OUT, "rpo_lstm_actor_sd_lstm.npz"), **{k: v for k, v in sd.items() if k.startswith("sd__lstm.")})
    made += ["rpo_lstm_actor.npz", "rpo_lstm_actor_sd_mlp.npz", "rpo_lstm_actor_sd_lstm.npz"]
    print("wrote", made)


if __name__ == "__main__":
    main()
