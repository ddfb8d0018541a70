"""`EKFLeeLanded`: sensor faults -> attitude EKF -> position/velocity Kalman filter -> waypoint logic -> Lee controller
on the ESTIMATES -> base-link wrench, every control step, for N envs, as a fixed chain of kernel launches.

Mirror of isaacgymenvs/tasks/ekf_lee_landed.py:308-530 (pre_physics_step) + :620-665.  The reference runs two Python
loops over envs per step (N x `EKF.update` in NumPy float64 after a D2H copy, N x `PVFilter` with ~40 tiny launches
each); here one step is:
  ozl_husky_step        target rides on the vehicle, x shift -0.08            (:628-629)
  ozl_apply_resets      reset_idx first, so the estimators see the re-spawned state   (:312-314)
  ozl_get_state         true root state [N,13]
  ozl_sensor_frontend   accel = dv/dt (+9.8 z), gyro, quaternion, pos, vel -- through the sensor-fault model after warm-up
  ozl_ekf_set_q         Q_state <- truth during warm-up / for reset envs        (:348-352)
  ozl_ekf_update        attitude EKF, float64                                   (:378-391)
  ozl_pv_reset/ozl_pv_step   PV filter: predict + gated position / velocity fixes (shared trigger counters)  (:353-358,417-444)
  ozl_waypoint_command  carrot waypoint + controller state                      (:458-503)
  ozl_lee_wrench        Lee position controller -> (m g * thrust, torque)       (:494-505)
  ozl_step_wrench       physics + observation + reward; wrench zeroed within 0.25 m of the target (:508-515)
Warm-up (`sim_step_count < ConvergenceTime` steps, :339): filters are fed the truth, the vehicle hovers on a constant
2.09 * 9.81 N force (:526-528).
"""
import torch

from .._lib import check, lib
from ..ahrs_ekf import EKFBank
from ..controllers import Controller, control
from ..pv_filter import PVFilterBank
from .landing import TARGET_Z, _VehicleTargetTask
from .ouzelum import _POMDP, refuse_multi_fault, x500_cfg_from_task


class EKFLeeLanded(_VehicleTargetTask):
    x_offset = -0.08                                   # ekf_lee_landed.py:629
    land_cutoff = 0.25                                 # ekf_lee_landed.py:508
    supports_states = False                            # the fused estimator step kernel has no states output
    supports_scenarios = False                         # ... and does not apply a scenario table
    supports_episode_log = False                       # ... and writes no episode records

    def __init__(self, cfg, *a, **k):
        env = cfg["env"]
        self.ConvergenceTime = env.get("ConvergenceTime", 300)              # cfg/task/EKFLeeLanded.yaml:18
        self.pos_sensor_freq = env.get("position_sensor_freq", 20)          # :21
        self.vel_sensor_freq = env.get("velocity_sensor_freq", 75)          # :22
        self.attach_pos_sensor = env.get("attach_pos_sensor", True)
        self.attach_vel_sensor = env.get("attach_vel_sensor", True)
        self._pomdp_mode = _POMDP[env.get("POMDP", "none")]
        self._pomdp_prob = float(env.get("pomdp_prob", 0.0))
        self.per_env_triggers = bool(env.get("perEnvSensorTriggers", False))
        self.fused = bool(env.get("fusedEstimator", True))      # one kernel for the whole estimator + controller chain
        self.fused_step = bool(env.get("fusedStep", True))      # ... and the vehicle + physics step in the same launch
        # the fused kernels can also write the estimated state [N,13] and the controller command [N,4] they computed (inspection /
        # parity tests: `_est`, `_cmd`); off by default -- 68 B per env of row-strided stores nobody on the step path reads
        self.expose_estimates = bool(env.get("exposeEstimates", False))
        super().__init__(cfg, *a, **k)

    def _native_cfg(self):
        # the observation itself also goes through the sensor-fault model env-side (ekf_lee_landed.py:659)
        # wrench_warmup_steps: during the estimator warm-up the hover force reaches every env and no landing is flagged (:508-529)
        refuse_multi_fault(type(self).__name__, self.cfg["env"])
        return x500_cfg_from_task(self.cfg, self.num_envs, target_fixed=1, die_z=self.die_z, plate_enable=1,
                                  plate_z=TARGET_Z, plate_radius=0.35, land_cutoff=self.land_cutoff,
                                  wrench_warmup_steps=int(self.ConvergenceTime))

    def create_sim(self):
        super().create_sim()
        n, dev = self.num_envs, self.device
        self.dt = float(self.cfg["sim"]["dt"])
        # envs of the whole job (all ranks): the reference's shared sensor-trigger counters advance once per env-iteration, so the
        # fix pattern depends on the TOTAL env count and the global env id, not on how the envs are sharded over GPUs
        self.num_envs_total = int(self.cfg["env"].get("numEnvsTotal", 0) or n)
        self.ekf = EKFBank(n, frequency=1 / self.dt, device=dev)            # :141
        self.pvfilters = PVFilterBank(n, [1.0, 1.0, 1.0], dev)              # :137: acc_var = 0.01 * 100
        self.controller = Controller(control(), dev)
        self.mg = 2.0 * (-float(self.cfg["sim"]["gravity"][2]))             # :459
        z = lambda *s: torch.zeros(*s, device=dev)
        self._root, self._est, self._cmd = z(n, 13), z(n, 13), z(n, 4)
        self._sensors, self.prev_root_linvels = z(n, 16), z(n, 3)
        self._q32, self._wrench = z(n, 4), z(n, 4)
        self.target_waypoints = z(n, 3)
        self._hover = z(n, 4)
        self._hover[:, 0] = -2.09 * float(self.cfg["sim"]["gravity"][2])    # :527
        self.sim_step_count = 0
        # shared trigger counters (ekf_lee_landed.py:153-154,425-440) => fix iff (step*N + env) % period == phase
        self._trigger = self._trigger_rule()
        self._seed, self._base = int(self.cfg["env"].get("seed", 0)), int(self.cfg["env"].get("envIdBase", 0))
        # fused path: argument block of ozl_ekf_lee_step (all pointers are fixed => the step is CUDA-graph capturable)
        import ctypes as C
        from .._lib import OzlEkfLeeArgs
        a = self._fa = OzlEkfLeeArgs()
        a.ekf_q4xN, a.ekf_P16xN = self.ekf._q.data_ptr(), self.ekf._P.data_ptr()
        a.pv_x9xN, a.pv_P81xN = self.pvfilters._x.data_ptr(), self.pvfilters._P.data_ptr()
        a.prev_linvel3, a.waypoint3 = self.prev_root_linvels.data_ptr(), self.target_waypoints.data_ptr()
        a.target3, a.reset, a.wrench4 = self.husky.target.data_ptr(), self.reset_buf.data_ptr() if hasattr(self, "reset_buf") else 0, self._wrench.data_ptr()
        a.est13 = self._est.data_ptr() if self.expose_estimates else None
        a.cmd4 = self._cmd.data_ptr() if self.expose_estimates else None
        a.gains16 = self.controller._gains
        a.dt, a.mg, a.hover_force = self.dt, self.mg, float(self._hover[0, 0].item())
        a.convergence_steps = int(self.ConvergenceTime)
        a.pomdp_mode, a.pomdp_prob = self._pomdp_mode, self._pomdp_prob
        pp, ph, vp, vh = self._trigger
        a.pos_period, a.pos_phase = (pp if self.attach_pos_sensor else 0), ph
        a.vel_period, a.vel_phase = (vp if self.attach_vel_sensor else 0), vh
        a.per_env_triggers = 1 if self.per_env_triggers else 0
        a.num_envs_total = self.num_envs_total
        a.acc_var[:] = [1.0, 1.0, 1.0]
        a.pos_var[:] = [0.0000001] * 3
        a.ekf_Dt, a.ekf_g_noise = float(self.ekf.Dt), float(self.ekf.g_noise)
        ctr = C.c_void_p()
        check(lib.ozl_step_counter_ptr(self.sim._h, C.byref(ctr)))
        self.husky.follow_step_counter(ctr.value)

    def _trigger_rule(self):
        def rule(freq, count0, attached):
            if not attached:
                return 0, 0
            # the counter starts at count0, a fix fires when count*dt > 1/freq and resets the counter to 0
            period = int((1.0 / freq) / self.dt + 1e-9) + 2          # first integer count with count*dt > 1/freq, plus the firing step
            k, cnt = 0, count0
            while not (cnt * self.dt > 1.0 / freq):
                cnt += 1
                k += 1
            return period, k % period
        pp, ph = rule(self.pos_sensor_freq, self.pos_sensor_freq * 0, self.attach_pos_sensor)
        vp, vh = rule(self.vel_sensor_freq, self.vel_sensor_freq / 2, self.attach_vel_sensor)
        return pp, ph, vp, vh

    def _launch(self, actions):
        if self.fused:
            return self._launch_fused()
        return self._launch_chain()

    def _launch_fused(self):
        """fusedStep: the whole control step in one launch; otherwise vehicle kernel -> fused estimator+controller kernel ->
        step kernel (three launches).  No host-changing arguments either way (CUDA-graph capturable)."""
        import ctypes as C
        self._fa.reset = self.reset_buf.data_ptr()
        if self.fused_step:
            # ONE launch: vehicle -> estimator + controller -> physics / observation / reward / reset (ozl_ekf_lee_landed_step)
            from .._lib import ptr
            ha = self.husky._a
            ha.reset = self.reset_buf.data_ptr()
            check(lib.ozl_ekf_lee_landed_step(self.sim._h, C.byref(self._fa), C.byref(ha), self.obs_buf.data_ptr(),
                                              self.rew_buf.data_ptr(), self.reset_buf.data_ptr(), self.progress_buf.data_ptr(),
                                              self._timeout_u8.data_ptr(), self.episode_return_buf.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream))
            self._target = self.husky.target
            self.sim_step_count += 1
            return
        self._target = self.husky.step(self.reset_buf)
        check(lib.ozl_ekf_lee_step(self.sim._h, C.byref(self._fa), torch.cuda.current_stream().cuda_stream))
        self.sim.step_wrench(self._wrench, self._target, self.obs_buf, self.rew_buf, self.reset_buf, self.progress_buf,
                             self._timeout_u8, self.episode_return_buf)
        self.sim_step_count += 1

    def _launch_chain(self):
        s = torch.cuda.current_stream().cuda_stream
        n = self.num_envs
        warm = self.sim_step_count < self.ConvergenceTime                              # :339
        self._target = self.husky.step(self.reset_buf)
        self.sim.apply_resets(self.reset_buf)                                          # :312-314
        self.sim.get_root(self._root)
        mode = 0 if warm else self._pomdp_mode
        check(lib.ozl_sensor_frontend(n, self._root.data_ptr(), self.prev_root_linvels.data_ptr(), self._sensors.data_ptr(),
                                      self.dt, mode, self._pomdp_prob, self._seed, self.sim_step_count, self._base, s))
        sens = self._sensors
        quat_true = self._root[:, 3:7].contiguous()
        self.ekf.set_q_from_root_quats(quat_true, None if warm else self.reset_buf)    # :348-352
        gyr, ang = sens[:, 3:6].contiguous(), sens[:, 6:10].contiguous()
        self.ekf.update(gyr, ang, ang_xyzw=True, q_f32_out=self._q32)                  # :378-391
        self.pvfilters.reset_states(self._root, self.reset_buf)                        # :353-358
        acc, pos, vel = sens[:, 0:3].contiguous(), sens[:, 10:13].contiguous(), sens[:, 13:16].contiguous()
        trig = self._trigger
        trig = (trig[0] if self.attach_pos_sensor else 0, trig[1], trig[2] if self.attach_vel_sensor else 0, trig[3])
        self.pvfilters.step(accels=acc, orientation=quat_true if warm else self._q32, dt=self.dt, flip_Qw=bool(warm),
                            gps_data=pos, gps_var=[0.0000001] * 3,                     # :408,430
                            vel_data=vel, vel_var=None,     # the reference's velocity fix runs with R = 0 (PVFilter.py:76-79)
                            trigger=trig,
                            iter_base=self.sim_step_count * self.num_envs_total + self._base)   # :417-444
        check(lib.ozl_waypoint_command(n, self._root.data_ptr(), self.pvfilters._x.data_ptr(), self._target.data_ptr(),
                                       self.target_waypoints.data_ptr(), 1 if warm else 0, self._est.data_ptr(),
                                       self._cmd.data_ptr(), s))                        # :458-503
        if warm:
            wrench = self._hover                                                        # :524-529
        else:
            wrench = self.controller.wrench(self._est, self._cmd, self.mg, out=self._wrench)
        self.sim.step_wrench(wrench, self._target, self.obs_buf, self.rew_buf, self.reset_buf, self.progress_buf,
                             self._timeout_u8, self.episode_return_buf)
        self.sim_step_count += 1

    # ---- checkpoint / resume: filter banks and glue buffers are part of the env state
    def state_dict(self):
        sd = super().state_dict()
        sd.update(ekf_q=self.ekf._q.cpu(), ekf_P=self.ekf._P.cpu(), pv_x=self.pvfilters._x.cpu(), pv_P=self.pvfilters._P.cpu(),
                  prev_root_linvels=self.prev_root_linvels.cpu(), target_waypoints=self.target_waypoints.cpu(),
                  sim_step_count=int(self.sim_step_count))
        return sd

    def load_state_dict(self, sd):
        super().load_state_dict(sd)
        self.ekf._q.copy_(sd["ekf_q"])
        self.ekf._P.copy_(sd["ekf_P"])
        self.pvfilters._x.copy_(sd["pv_x"])
        self.pvfilters._P.copy_(sd["pv_P"])
        self.prev_root_linvels.copy_(sd["prev_root_linvels"])
        self.target_waypoints.copy_(sd["target_waypoints"])
        self.sim_step_count = int(sd["sim_step_count"])

    @property
    def landings(self):
        return int(self.sim.metrics()[2].item())

    @property
    def resets(self):
        """The reference's `self.epi` (ekf_lee_landed.py:316): number of env resets applied, the initial one included."""
        return int(self.sim.metrics()[15].item())

    def write_metrics(self, log_dir):
        """The two files an EKFLeeLanded evaluation run leaves behind (ekf_lee_landed.py:319-331), from the device-side episode
        statistics (one host read when called, instead of two file writes inside every step):
          <log_dir>/metrics/<pomdp>_<prob>_ep_count.txt   resets applied so far (`self.epi`)
          <log_dir>/metrics/<pomdp>_<prob>.txt            episodes that ended after the vehicle was reached (`self.Landoa`)"""
        import os
        env = self.cfg["env"]
        tag = f"{env.get('POMDP', 'none')}_{float(env.get('pomdp_prob', 0.0))}"
        os.makedirs(os.path.join(log_dir, "metrics"), exist_ok=True)
        m = self.sim.metrics().cpu()
        with open(os.path.join(log_dir, "metrics", f"{tag}_ep_count.txt"), "w") as f:
            f.write(str(int(m[15])))
        with open(os.path.join(log_dir, "metrics", f"{tag}.txt"), "w") as f:
            f.write(str(int(m[2])))
        return int(m[2]), int(m[15])

    @property
    def episodes(self):
        return int(self.sim.metrics()[9].item())
