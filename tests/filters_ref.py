"""ctypes front end of `tests/filters_ref.c`, the exact CPU twin of the estimators in ouzelum_b200/csrc/filters.cuh.

Two shared objects are built from the one source with gcc (`-O2 -ffp-contract=off -fno-fast-math`, plus `-mfma` where the host
has FMA3, the flags of oracle/c_oracle.py):
  * float32 (`F32`): the bit-exact twin of `pv_step_kernel`, `ekf_update_kernel` and the filter stages of `ekf_lee_fused_kernel`
  * float64 (`F64`): the same operation sequence with the PV scalar type switched to double -- the high-precision reference
They go to oracle/_build/ (git-ignored) when that directory is writable, else to a per-user temporary directory.

Arrays are numpy in / numpy out in the plane layouts of the device banks: x [9][N], P [81][N], EKF q [4][N], EKF P [16][N]; per-env
inputs are row-major [N, k].  `PVTwinBank` / `EKFTwinBank` wrap the drivers behind the interfaces of the oracle banks.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "filters_ref.c")

G_NOISE = 0.3 ** 2            # ahrs_ekf.py:1004
S_EPS = 0.0000001             # ahrs_ekf.py:1332, the constant ozl_ekf_update passes


def _out_dir():
    d = os.path.join(ROOT, "oracle", "_build")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), f"ozl_filters_ref_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


def build(f64=False, force=False):
    out = os.path.join(_out_dir(), "libfilters_ref_f64.so" if f64 else "libfilters_ref_f32.so")
    if not force and os.path.exists(out) and os.path.getmtime(out) > os.path.getmtime(SRC):
        return out
    try:
        has_fma = " fma " in open("/proc/cpuinfo").read()
    except OSError:
        has_fma = False
    tmp = f"{out}.{os.getpid()}.tmp"
    cmd = ["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math"] + (["-mfma"] if has_fma else []) + \
          (["-DFILTERS_REF_F64"] if f64 else []) + ["-fopenmp", "-shared", "-fPIC", "-o", tmp, SRC, "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("gcc failed: " + r.stderr)
    os.replace(tmp, out)
    return out


_LIBS = {}


def _lib(dtype):
    dtype = np.dtype(dtype)
    if dtype not in _LIBS:
        f64 = dtype == np.float64
        lib = C.CDLL(build(f64))
        assert lib.ozl_ref_real_size() == dtype.itemsize
        lib.ozl_ref_pv_step.restype = None
        lib.ozl_ref_pv_step.argtypes = [C.c_int64] + [C.c_void_p] * 8 + [C.c_double] + [C.c_void_p] * 3 + [C.c_int] * 4 + \
                                       [C.c_uint32] * 4 + [C.c_uint64]
        lib.ozl_ref_ekf_update.restype = None
        lib.ozl_ref_ekf_update.argtypes = [C.c_int64] + [C.c_void_p] * 4 + [C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p]
        _LIBS[dtype] = lib
    return _LIBS[dtype]


def coop_worker_counts(n, steps, trigger, per_env=False, env_id_base=0, n_total=None):
    """Worker counts S of the two cooperative fix passes of ekf_lee_fused_kernel (pv_correct_coop) over `steps` steps, from the
    trigger rule alone: per warp of valid lanes (nl of them, the last warp of the launch a prefix), S = min(9, floor((nl + 0.5) /
    jobs)), where the jobs of pass 1 are the envs with any fix and those of pass 2 the envs with both.  Returns (set, set)."""
    n_total = int(n_total or n)
    pp, ph, vp, vh = trigger
    ids = np.arange(n, dtype=np.int64) + int(env_id_base)
    s1, s2 = set(), set()
    for t in range(steps):
        k = np.full(n, t, np.int64) if per_env else t * n_total + ids
        fp = (k % pp == ph) if pp else np.zeros(n, bool)
        fv = (k % vp == vh) if vp else np.zeros(n, bool)
        for w0 in range(0, n, 32):
            nl = min(32, n - w0)
            for jobs, s in ((int((fp | fv)[w0:w0 + 32].sum()), s1), (int((fp & fv)[w0:w0 + 32].sum()), s2)):
                if jobs:
                    s.add(min(9, (2 * nl + 1) // (2 * jobs)))
    return s1, s2


def _arr(a, dtype, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(np.asarray(a), dtype=dtype)
    if shape is not None:
        assert a.shape == shape, (a.shape, shape)
    return a


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pv_step(x9, P81, accel=None, quat=None, pos_meas=None, vel_meas=None, pos_mask=None, vel_mask=None, dt=0.01,
            acc_var=(1.0, 1.0, 1.0), pos_var=None, vel_var=None, flip_qw=True, trigger=None, iter_base=0, dtype=np.float32):
    """One pv_step_kernel launch: returns new (x9 [9,N], P81 [81,N]) in `dtype`.  Predict runs when `accel` is given; a fix runs
    where its mask is set or, without a mask, where (iter_base + i) % period == phase with trigger = (pos_period, pos_phase,
    vel_period, vel_phase) (default: every env takes a supplied measurement).  pos_var / vel_var None: R = 0."""
    lib = _lib(dtype)
    x9 = np.array(x9, dtype=dtype, order="C")
    P81 = np.array(P81, dtype=dtype, order="C")
    n = x9.shape[1]
    assert x9.shape == (9, n) and P81.shape == (81, n)
    ins = [_arr(accel, dtype, (n, 3)), _arr(quat, dtype, (n, 4)), _arr(pos_meas, dtype, (n, 3)), _arr(vel_meas, dtype, (n, 3)),
           _arr(pos_mask, np.uint8, (n,)), _arr(vel_mask, np.uint8, (n,))]
    av = _arr(acc_var, dtype, (3,))
    pv = _arr(pos_var if pos_var is not None else np.zeros(3), dtype, (3,))
    vv = _arr(vel_var if vel_var is not None else np.zeros(3), dtype, (3,))
    trig = (1, 0, 1, 0) if trigger is None else tuple(int(v) for v in trigger)
    lib.ozl_ref_pv_step(n, _p(x9), _p(P81), *[_p(a) for a in ins], float(dt), _p(av), _p(pv), _p(vv),
                        int(pos_var is not None), int(vel_var is not None), int(bool(flip_qw)), int(accel is not None),
                        *trig, int(iter_base))
    return x9, P81


def ekf_update(q4, P16, gyr, ang, ang_xyzw=False, Dt=0.01, g_noise=G_NOISE, q_f32_out=False):
    """One ekf_update_kernel launch (float64 state, float32 sensors): returns new (q4 [4,N], P16 [16,N]) and, with q_f32_out,
    the float32 copy of q [N,4] as third element."""
    lib = _lib(np.float32)
    q4 = np.array(q4, dtype=np.float64, order="C")
    P16 = np.array(P16, dtype=np.float64, order="C")
    n = q4.shape[1]
    assert q4.shape == (4, n) and P16.shape == (16, n)
    g = _arr(gyr, np.float32, (n, 3))
    a = _arr(ang, np.float32, (n, 4))
    qf = np.zeros((n, 4), np.float32) if q_f32_out else None
    lib.ozl_ref_ekf_update(n, _p(q4), _p(P16), _p(g), _p(a), int(bool(ang_xyzw)), float(Dt), float(g_noise), S_EPS, _p(qf))
    return (q4, P16, qf) if q_f32_out else (q4, P16)


class PVTwinBank:
    """The interface of oracle.pv_filter.PVFilterBank (state [N,9], cov [N,9,9], prediction_step, correction_step) on the C twin."""

    def __init__(self, n, acc_var, dtype=np.float32):
        self.f, self.n = dtype, n
        self.state = np.zeros((n, 9), dtype=dtype)
        self.cov = np.broadcast_to(np.eye(9, dtype=dtype) * dtype(1000), (n, 9, 9)).copy()
        self.acc_var = np.asarray(acc_var, dtype=dtype)

    def _step(self, **kw):
        x, P = pv_step(self.state.T, self.cov.reshape(self.n, 81).T, acc_var=self.acc_var, dtype=self.f, **kw)
        self.state, self.cov = np.ascontiguousarray(x.T), np.ascontiguousarray(P.T).reshape(self.n, 9, 9)

    def prediction_step(self, accels, orientation, dt, flip_Qw=True, mask=None):
        assert mask is None
        self._step(accel=accels, quat=orientation, dt=dt, flip_qw=flip_Qw)

    def correction_step(self, gps_data=None, gps_var=None, vel_data=None, vel_var=None, mask=None):
        """PVFilter.py:67-110 semantics: the velocity fix has R = 0 unless *gps_var* is given; velocity fix first, as the oracle."""
        m = np.ones(self.n, bool) if mask is None else np.asarray(mask, bool)
        if vel_data is not None:
            self._step(vel_meas=vel_data, vel_mask=m, vel_var=None if gps_var is None else vel_var)
        if gps_data is not None:
            self._step(pos_meas=gps_data, pos_mask=m, pos_var=gps_var)


class EKFTwinBank:
    """The attitude EKF of the glue (oracle.ekf_lee_landed.EKFLeeGlue.ekf) on the C twin.  The glue hands `update` the quaternion
    it normalised with np.linalg.norm; the kernel normalises the stored one itself, so the twin reads the glue's raw `Q` instead."""

    def __init__(self, glue, n, Dt=0.01, g_noise=G_NOISE):
        self.glue, self.n = glue, n
        self.Dt, self.g_noise = float(Dt), float(g_noise)
        self.P = np.broadcast_to(np.identity(4), (n, 4, 4)).copy()

    def update(self, q_normalised, gyr, ang):
        del q_normalised
        g32, a32 = np.asarray(gyr).astype(np.float32), np.asarray(ang).astype(np.float32)
        assert np.array_equal(g32, gyr) and np.array_equal(a32, ang)          # the float32 sensors, widened
        q4, P16 = ekf_update(self.glue.Q.T, self.P.reshape(self.n, 16).T, g32, a32, ang_xyzw=False, Dt=self.Dt,
                             g_noise=self.g_noise)
        self.P = np.ascontiguousarray(P16.T).reshape(self.n, 4, 4)
        return np.ascontiguousarray(q4.T)
