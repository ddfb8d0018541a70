"""Classical-control baseline task: the Lee position controller flies the x500 through a base-link wrench.

Mirror of isaacgymenvs/tasks/lee_landed.py:263-330: actions are ignored; every step
  target = (0, 0, 1, yaw 0)                                                     (lee_landed.py:299-302)
  thrust, torque = Controller(root_states, target)                               (:311)
  forces[:, 0, 2] = (2 * 9.81) * thrust ; torques[:, 0] = torque                  (:296,313-314)
  zero wrench within 0.2 m of the controller target (landing flag)                (:318-322)
ONE launch per step (`ozl_lee_landed_step`: vehicle, controller on the re-spawned true state, landing detector on the controller
target, physics / observation / reward); `env.fusedStep = False` keeps the chain vehicle -> apply_resets -> state gather ->
`ozl_lee_wrench` -> `ozl_step_wrench` for A/B tests.
"""
import torch

from ..controllers import Controller, control
from .landing import TARGET_Z, _VehicleTargetTask
from .ouzelum import x500_cfg_from_task


class LeeLanded(_VehicleTargetTask):
    land_cutoff = 0.2                                                  # lee_landed.py:318
    vehicle_moves = True

    def _native_cfg(self):
        # the landing detector of this task measures the distance to the CONTROLLER target (0,0,1), which is also what the
        # stored target is set to below; the reward's target rides on the Husky (post_physics_step, lee_landed.py:339-340)
        # (the detector distance is measured to the controller target: the step kernels take it as `det_tgt`)
        return x500_cfg_from_task(self.cfg, self.num_envs, target_fixed=1, die_z=self.die_z, plate_enable=1,
                                  plate_z=TARGET_Z, plate_radius=0.35,
                                  land_cutoff=self.land_cutoff if bool(self.cfg["env"].get("fusedStep", True)) else 0.0)

    def _check_scenarios(self, rows):
        from .._lib import SCENARIO_LAYOUT
        if not torch.isnan(rows[:, SCENARIO_LAYOUT["OZL_SCN_FAULT_ROTOR"]]).all():
            raise ValueError("LeeLanded: scenario rows must leave the fault group NaN (the steps are wrench-actuated: rotor faults "
                             "do not apply)")

    def create_sim(self):
        super().create_sim()
        self.controller = Controller(control(), self.device)
        self.mg = 2.0 * (-float(self.cfg["sim"]["gravity"][2]))        # lee_landed.py:296
        self._cmd = torch.zeros(self.num_envs, 4, device=self.device)
        self._cmd[:, 2] = 1.0                                          # lee_landed.py:301-302
        self._root = torch.empty(self.num_envs, 13, device=self.device)
        self._wrench = torch.empty(self.num_envs, 4, device=self.device)
        self._landed_chain = torch.zeros(self.num_envs, dtype=torch.bool, device=self.device)
        from .._lib import OzlLeeLandedArgs
        a = self._la = OzlLeeLandedArgs()
        a.gains16 = self.controller._gains
        a.cmd[:] = [0.0, 0.0, 1.0, 0.0]                                # lee_landed.py:299-302
        a.mg = self.mg
        a.wrench4 = self._wrench.data_ptr()

    @property
    def landed_flag(self):
        """Per env: came within 0.2 m of the controller target during the current episode (lee_landed.py:318-320 keeps ONE Python
        bool for all envs; here the flag is per env, bit 31 of the env's fault word)."""
        if not bool(self.cfg["env"].get("fusedStep", True)):
            return self._landed_chain
        _, fault = self.sim.get_params()
        return fault[:, 1] < 0

    def _launch(self, actions):
        import ctypes as C
        from .._lib import check, lib
        s = torch.cuda.current_stream().cuda_stream
        if bool(self.cfg["env"].get("fusedStep", True)):
            check(lib.ozl_lee_landed_step(self.sim._h, C.byref(self._la), C.byref(self.husky._a), self.obs_buf.data_ptr(),
                                          self.rew_buf.data_ptr(), self.reset_buf.data_ptr(), self.progress_buf.data_ptr(),
                                          self._timeout_u8.data_ptr(), self.episode_return_buf.data_ptr(), s))
            self._target = self.husky.target
            return
        self._target = self.husky.step(self.reset_buf)
        self.sim.apply_resets(self.reset_buf)                          # reset_idx precedes the controller (lee_landed.py:267-270)
        check(lib.ozl_get_state(self.sim._h, self._root.data_ptr(), None, None, None, s))
        # NOTE reset envs: the reference runs the controller on the freshly re-spawned state (reset_idx precedes it,
        # lee_landed.py:267-270) and then zeroes their forces (:325-326); the step kernel zeroes the wrench of reset envs too.
        self.controller.wrench(self._root, self._cmd, self.mg, out=self._wrench)
        # landing detector on the controller target (lee_landed.py:305,318-322)
        near = (self._cmd[:, 0:3] - self._root[:, 0:3]).norm(dim=1) < self.land_cutoff
        self._landed_chain |= near
        self._wrench.masked_fill_(near[:, None], 0.0)
        self.sim.step_wrench(self._wrench, self._target, self.obs_buf, self.rew_buf, self.reset_buf, self.progress_buf,
                             self._timeout_u8, self.episode_return_buf)
