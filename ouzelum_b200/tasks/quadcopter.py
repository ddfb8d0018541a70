"""`Quadcopter`: the stock NVIDIA hover task (BASELINE config 1) as one fused kernel per step.

Mirror of isaacgymenvs/tasks/quadcopter.py (12 actions: 8 rotor-tilt joint rates + 4 thrust rates; 21 observations).
The reference builds a 9-body MJCF articulation and lets PhysX drive 8 PD joints; here the vehicle is one rigid body
with four kinematically tilting thrust vectors (`ozl_quadcopter_step`).  Observation / reward / reset arithmetic follows
quadcopter.py:359-418 exactly; the dynamics are a documented stand-in (parity unpinned, SURVEY 8a row Q).
"""
import ctypes as C
import math

import torch

from .._lib import OzlQuadcopterArgs, check, lib
from ..vec_task import VecTask
from .ouzelum import asymmetric_states, refuse_multi_fault


def vehicle_constants():
    """Composite rigid body of the procedurally built vehicle (quadcopter.py:121-202) at zero tilt."""
    pi = math.pi
    chassis_radius, chassis_thickness, rotor_radius, rotor_thickness, rotor_arm_radius = 0.1, 0.03, 0.04, 0.01, 0.01
    m_c = pi * chassis_radius ** 2 * chassis_thickness * 50          # density attributes, quadcopter.py:150,174,192
    m_a = 4.0 / 3.0 * pi * rotor_arm_radius ** 3 * 200
    m_r = pi * rotor_radius ** 2 * rotor_thickness * 1000
    ra = chassis_radius + 0.25 * rotor_arm_radius
    rr = ra + rotor_radius + 0.25 * rotor_arm_radius
    ixx = m_c * (3 * chassis_radius ** 2 + chassis_thickness ** 2) / 12 + 4 * (0.4 * m_a * rotor_arm_radius ** 2) + 2 * m_a * ra ** 2 \
        + 4 * (m_r * (3 * rotor_radius ** 2 + rotor_thickness ** 2) / 12) + 2 * m_r * rr ** 2
    izz = 0.5 * m_c * chassis_radius ** 2 + 4 * (0.4 * m_a * rotor_arm_radius ** 2) + 4 * m_a * ra ** 2 \
        + 4 * (0.5 * m_r * rotor_radius ** 2) + 4 * m_r * rr ** 2
    return dict(mass=m_c + 4 * m_a + 4 * m_r, ixx=ixx, iyy=ixx, izz=izz)


class Quadcopter(VecTask):
    def __init__(self, cfg, rl_device, sim_device, graphics_device_id, headless, virtual_screen_capture=False, force_render=False):
        self.cfg = cfg
        self.max_episode_length = self.cfg["env"]["maxEpisodeLength"]
        self.debug_viz = self.cfg["env"].get("enableDebugVis", False)
        self.cfg["env"]["numObservations"] = 21          # quadcopter.py:57-60
        self.cfg["env"]["numActions"] = 12
        asymmetric_states(type(self).__name__, self.cfg["env"], supported=False)      # its 21-obs vehicle has no states output
        refuse_multi_fault(type(self).__name__, self.cfg["env"])
        super().__init__(config=self.cfg, rl_device=rl_device, sim_device=sim_device, graphics_device_id=graphics_device_id,
                         headless=headless, virtual_screen_capture=virtual_screen_capture, force_render=force_render)
        self._timeout_u8 = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
        self.timeout_buf = self._timeout_u8.view(torch.bool)

    supports_episode_log = False       # its step kernel writes no episode records

    def set_scenarios(self, rows):
        raise ValueError("Quadcopter: scenario tables are not supported (its step kernel does not apply them)")

    def enable_episode_log(self, capacity):
        raise ValueError("Quadcopter: the episode log is not supported (its step kernel writes no records)")

    def create_sim(self):
        n, dev = self.num_envs, self.device
        env, sim = self.cfg["env"], self.cfg.get("sim", {})
        self.dt = float(sim.get("dt", 0.01))
        self.root_states = torch.zeros(n, 13, device=dev)
        self.root_states[:, 2] = 1.0                     # default_pose.p.z = 1.0, quadcopter.py:232-233
        self.root_states[:, 6] = 1.0
        self.root_positions, self.root_quats = self.root_states[:, 0:3], self.root_states[:, 3:7]
        self.root_linvels, self.root_angvels = self.root_states[:, 7:10], self.root_states[:, 10:13]
        self.dof_positions = torch.zeros(n, 8, device=dev)
        self.dof_position_targets = torch.zeros(n, 8, device=dev)
        self.thrusts = torch.zeros(n, 4, device=dev)
        a = self._a = OzlQuadcopterArgs()
        a.n = n
        a.root13, a.dof_pos8, a.dof_target8 = self.root_states.data_ptr(), self.dof_positions.data_ptr(), self.dof_position_targets.data_ptr()
        a.thrust4 = self.thrusts.data_ptr()
        a.seed, a.env_id_base = int(env.get("seed", 0)), int(env.get("envIdBase", 0))
        a.max_episode_length, a.substeps = int(env["maxEpisodeLength"]), int(sim.get("substeps", 2))
        a.dt, a.gravity_z = self.dt, float(sim.get("gravity", [0, 0, -9.81])[2])
        a.clip_actions = float(min(env.get("clipActions", math.inf), 3.0e38))
        a.clip_obs = float(min(env.get("clipObservations", math.inf), 3.0e38))
        vc = vehicle_constants()
        a.mass, a.ixx, a.iyy, a.izz = vc["mass"], vc["ixx"], vc["iyy"], vc["izz"]
        # the RNG's time axis lives in a DEVICE step-counter record the kernel reads and advances itself, so a step takes no
        # host-changing argument and can be replayed from a CUDA graph (env.useCudaGraph)
        self._step_record = torch.zeros(2, dtype=torch.int64, device=dev)
        check(lib.ozl_step_record_init(self._step_record.data_ptr(), n, 0, torch.cuda.current_stream().cuda_stream))
        a.step_record = self._step_record.data_ptr()
        self.use_cuda_graph = bool(env.get("useCudaGraph", False))
        self._graph, self._static_actions = None, None

    @property
    def step_count(self):
        out = C.c_uint64()
        check(lib.ozl_step_record_read(self._step_record.data_ptr(), C.byref(out), torch.cuda.current_stream().cuda_stream))
        return out.value

    def _launch(self, actions):
        a = self._a
        a.actions12, a.obs21, a.rew = actions.data_ptr(), self.obs_buf.data_ptr(), self.rew_buf.data_ptr()
        a.reset, a.progress, a.timeout = self.reset_buf.data_ptr(), self.progress_buf.data_ptr(), self._timeout_u8.data_ptr()
        check(lib.ozl_quadcopter_step(C.byref(a), torch.cuda.current_stream().cuda_stream))

    def _fused_step(self, actions):
        if not self.use_cuda_graph:
            self._launch(actions)
            return
        if self._graph is None:
            self._static_actions = torch.empty_like(actions)
            self._static_actions.copy_(actions)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._launch(self._static_actions)
            self._graph = g
        self._static_actions.copy_(actions)
        self._graph.replay()

    def reset_idx(self, env_ids):
        self.reset_buf[env_ids] = 1                      # applied inside the next step's kernel (quadcopter.py:304-306)
