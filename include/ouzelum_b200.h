/*
 * ouzelum_b200 -- C ABI of the B200-native quadcopter env-step path.
 *
 * This is the drop-in boundary: what the reference reaches through the Isaac Gym pybind API
 * (gymapi / gymtorch -- a closed binary that is NOT under the reference tree) plus the eager
 * torch ops around it.  Every entry point below names the reference interface it replaces
 * (paths relative to the reference checkout root).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; device pointers are ordinary pointers into CUDA global memory that the
 *     CALLER owns (torch tensors on the Python side: pass tensor.data_ptr()).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  No entry point on
 *     the step path synchronises with the host or allocates; everything is CUDA-graph capturable.
 *   - every function returns 0 on success, non-zero on error; ozl_last_error() returns a
 *     thread-local message for the last failing call.
 *   - quaternions in root states are xyzw (Isaac Gym); linear AND angular velocity are world-frame.
 *   - handles are not thread-safe; distinct handles are independent.  One process per GPU.
 */
#ifndef OUZELUM_B200_H
#define OUZELUM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OZL_ABI_VERSION 7   /* 3: ozl_cfg.dr[] (domain-randomisation schema), per-env yaw_km (params8), wrench_warmup_steps,
                               ozl_ekf_lee_args.num_envs_total, i64 reset mirror in ozl_host_io
                               4: (additive) ozl_metrics_xchg_* / ozl_metrics_push / ozl_metrics_sum, ozl_noise_lambda_apply
                               5: (additive) ozl_set_states_output, OZL_STATE_* layout of the privileged critic state
                               6: (additive) ozl_set_scenarios, OZL_SCN_* layout of a scenario row
                               7: (additive) fault_mode 2 (multi-rotor and gradual rotor faults): ozl_cfg.fault_rotors_lo / _hi /
                                  fault_ramp_steps in the former reserved0 / reserved1 (same size), ozl_get_rotor_eff /
                                  ozl_set_rotor_eff, scenario group OZL_SCN_RFAULT_*
                                  (additive, still 7) ozl_set_episode_log, OZL_EPLOG_* layout of an episode record */

/* sensor-fault model of isaacgymenvs/utils/POMDP.py:4-42 */
enum { OZL_POMDP_NONE = 0, OZL_POMDP_FLICKER = 1, OZL_POMDP_NOISE = 2, OZL_POMDP_FLICKER_NOISE = 3 };

/* Domain randomisation of one per-env parameter, drawn when the env is reset.  Schema of the reference's
 * `randomization_params` (isaacgymenvs/utils/dr_utils.py:71-132 generate_random_samples, applied at resets only,
 * tasks/base/vec_task.py:538-768):
 *   distribution  uniform: range = (lo, hi) ; loguniform: exp(U(log lo, log hi)) ; gaussian: range = (mu, sigma)
 *   operation     scaling: param = nominal * sample ; additive: param = nominal + sample
 *   schedule      none ; linear: s = min(step, schedule_steps) / schedule_steps ; constant: s = step < schedule_steps ? 0 : 1
 *                 additive: range *= s ; scaling: lo/hi/mu -> x*s + (1-s), sigma -> sigma*s     (dr_utils.py:82-131)
 * `step` is the handle's step counter (the reference's gym frame count).  Draws are Philox words keyed by (seed, global env id,
 * step): word j of P_DR0|P_DR1 for parameter j (and word j of P_DR2|P_DR3 as the second uniform of a gaussian). */
enum { OZL_DR_NONE = 0, OZL_DR_UNIFORM = 1, OZL_DR_LOGUNIFORM = 2, OZL_DR_GAUSSIAN = 3 };
enum { OZL_DR_SCALING = 0, OZL_DR_ADDITIVE = 1 };
enum { OZL_DR_SCHED_NONE = 0, OZL_DR_SCHED_LINEAR = 1, OZL_DR_SCHED_CONSTANT = 2 };
enum { OZL_DR_MASS = 0, OZL_DR_IXX = 1, OZL_DR_IYY = 2, OZL_DR_IZZ = 3, OZL_DR_ARM = 4, OZL_DR_THRUST_SCALE = 5, OZL_DR_YAW_KM = 6,
       OZL_DR_NUM = 7 };
typedef struct ozl_dr_param {
    int32_t distribution;         /* OZL_DR_NONE / _UNIFORM / _LOGUNIFORM / _GAUSSIAN */
    int32_t operation;            /* OZL_DR_SCALING / _ADDITIVE */
    float range[2];               /* (lo, hi) or (mu, sigma) */
    int32_t schedule;             /* OZL_DR_SCHED_* */
    int32_t schedule_steps;
} ozl_dr_param;

/* Task configuration.  Defaults (ozl_cfg_default) reproduce isaacgymenvs/cfg/task/Ouzelum.yaml and
 * the literals in isaacgymenvs/tasks/ouzelum.py; the "extras" are zero-default options with no
 * reference counterpart (SURVEY.md section 8a row P). */
typedef struct ozl_cfg {
    int32_t abi_version;          /* must be OZL_ABI_VERSION */
    int16_t fault_rotors_lo;      /* fault_mode 2: number of faulted rotors drawn in [lo, hi], 0 <= lo <= hi <= 4 (default 1, 1);  */
    int16_t fault_rotors_hi;      /* these two and fault_ramp_steps sit in what were reserved words, so sizeof(ozl_cfg) is unchanged */
    int64_t num_envs;             /* envs simulated by THIS handle (the local shard)            cfg env.numEnvs */
    int64_t env_id_base;          /* global id of local env 0: RNG is keyed by global id, so results do not depend on the sharding */
    uint64_t seed;
    int32_t max_episode_length;   /* env.maxEpisodeLength (2000)                                  Ouzelum.yaml:10 */
    int32_t target_period;        /* resample the target when progress % period == 0 (500)        ouzelum.py:221  */
    int32_t target_fixed;         /* 1: never resample (landing-family tasks drive the target)                    */
    int32_t substeps;             /* sim.substeps (2)                                             Ouzelum.yaml:21 */
    int32_t control_freq_inv;     /* env.controlFrequencyInv (1)                                  vec_task.py:100 */
    float dt;                     /* sim.dt (0.01)                                                Ouzelum.yaml:20 */
    float gravity_z;              /* -9.81                                                        ouzelum.py:118  */
    float clip_actions;           /* env.clipActions (1.0)                                        vec_task.py:327 */
    float clip_obs;               /* env.clipObservations (5.0)                                   vec_task.py:353 */
    float thrust_rate;            /* dt * 2000                                                    ouzelum.py:237  */
    float thrust_max;             /* 2000                                                         ouzelum.py:91   */
    float die_dist;               /* 8.0                                                          ouzelum.py:326  */
    float die_z;                  /* 0.5 (0.3 for the landing family)                             ouzelum.py:327  */
    float up_coef;                /* 5.0 (1.0 for Quadcopter)                                     ouzelum.py:314  */
    float spawn_base[3];          /* (0,0,1)                                                      ouzelum.py:150  */
    float spawn_lo[3];            /* (-1.5,-1.5,-0.2)                                             ouzelum.py:207  */
    float spawn_range[3];         /* (3.0,3.0,1.7)                                                                */
    float target_scale[3];        /* (10,10,1)                                                    ouzelum.py:183  */
    float target_off[3];          /* (-5,-5,1)                                                                    */
    /* single-rigid-body x500 (assets/x500/x500.urdf, SURVEY 8a row P) */
    float mass, ixx, iyy, izz, arm, com_z, max_angvel;
    /* extras (no reference counterpart; 0 => reference behaviour) */
    float lin_drag;               /* F = -k v (world)                                                             */
    float yaw_km;                 /* rotor reaction torque about body z per newton of thrust                      */
    int32_t fault_mode;           /* 1: single-rotor loss of effectiveness, schedule drawn at reset
                                     2: multi-rotor and gradual loss of effectiveness (see "Rotor faults, mode 2" below) */
    float fault_eff_lo, fault_eff_range;
    int32_t dr_enable;            /* 1: randomise the per-env parameters at reset according to dr[]               */
    ozl_dr_param dr[7];           /* indexed by OZL_DR_*; default: mass/Ixx/Iyy/Izz/arm/thrust-scale = scaling x uniform
                                     [0.8, 1.2) (dr_utils.py:121-130), yaw_km = none                              */
    int32_t pomdp_mode;           /* OZL_POMDP_* applied to the observation inside the step (tasks/landed.py:340) */
    float pomdp_prob;             /* flicker probability                                          POMDP.py:8      */
    float noise_sigma;            /* multiplicative noise U(1-s, 1+s)                             POMDP.py:9-10   */
    int32_t collect_metrics;      /* 1: accumulate the episode/reward metrics vector (ozl_metrics_read)           */
    int32_t plate_enable;         /* 1: inelastic landing plate under the target (landing family; new, see DESIGN) */
    float plate_z;                /* plate height (0.377 = Husky top plate, landing.py:76)                        */
    float plate_radius;           /* horizontal reach of the plate around the target                              */
    float land_cutoff;            /* >0: zero the wrench within this distance of the target and flag a landing
                                     (tasks/landed.py:288-295 0.2, lee_landed.py:318-322 0.2, ekf_lee_landed.py:508-515 0.25) */
    int32_t wrench_warmup_steps;  /* wrench-actuated steps with step counter < this value are the estimator warm-up of
                                     tasks/ekf_lee_landed.py:339,508-529: the wrench reaches EVERY env (no near-target cut, no
                                     zeroing for just-reset envs) and the landing flag is not raised.  0 = no warm-up      */
    int32_t fault_ramp_steps;     /* fault_mode 2: steps over which the loss ramps in, 0 <= ramp < 2^24 (0 or 1: abrupt; default 0) */
} ozl_cfg;

/* Rotor faults, mode 2 (cfg.fault_mode = 2, "multi").  At every reset of env i, with Philox words keyed by (seed, global env id,
 * step, purpose) like every other draw -- r0..r2 of the P_FAULT draw that mode 1 uses, w0..w3 of one more draw (P_RFAULT) --
 *   k      = fault_rotors_lo + umulhi(r2, fault_rotors_hi - fault_rotors_lo + 1)          number of faulted rotors
 *   rotors = the first k entries of permutation umulhi(r0, 24) of {0,1,2,3}, the 24 in lexicographic order
 *   e_j    = fault_eff_lo + fault_eff_range * u01(w_j) for a faulted rotor j, 1.0f for a healthy one
 *   onset  = umulhi(r1, max_episode_length) (mode 1's onset), or never (0x1FFFFFFF) when k = 0
 * At progress p >= onset (progress after the reset phase of the step), with d = p - onset, rotor j's force is multiplied by
 *   a_j = e_j                                                    if fault_ramp_steps <= 1 or d + 1 >= fault_ramp_steps
 *   a_j = fmaf((float)(d + 1) * inv_ramp, e_j - 1.0f, 1.0f)      otherwise, inv_ramp = (float)(1.0 / fault_ramp_steps)
 * (a healthy rotor gets exactly 1).  The fault is active (metrics slot 14) while p >= onset; OZL_STATE_EFF .. +3 report a_j (1 on
 * wrench-actuated steps, where no fault is applied).  e_0..e_3 live in a per-env plane of the handle (ozl_get_rotor_eff /
 * ozl_set_rotor_eff), the onset in the fault word (ozl_get_params fault2[:, 1]; the rotor id and the params8 effectiveness are
 * unused).  Mode 2 applies on ozl_step, ozl_step_tracking, ozl_step_wrench, ozl_step_host*, ozl_landing_step,
 * ozl_apply_resets and the initial state (no fault); ozl_rollout, ozl_lee_landed_step and ozl_ekf_lee_landed_step refuse to run.
 * ozl_create checks 0 <= lo <= hi <= 4, 0 <= fault_ramp_steps < 2^24, fault_eff_lo in [0, 1] and fault_eff_lo + fault_eff_range
 * in [fault_eff_lo, 1]. */

typedef struct ozl_env ozl_env;   /* opaque */

/* Fill *cfg with the Ouzelum defaults for `num_envs` envs.  (cfg/task/Ouzelum.yaml, tasks/ouzelum.py:42-99) */
int ozl_cfg_default(ozl_cfg* cfg, int64_t num_envs);

/* Create the private SoA state for cfg->num_envs envs on CUDA device `device`.
 * Replaces: VecTask.__init__ -> create_sim/_create_envs (tasks/ouzelum.py:112-178; an O(N) Python loop
 * of gym.create_env/create_actor) + acquire/wrap of the root-state tensors (tasks/ouzelum.py:59-99). */
int ozl_create(const ozl_cfg* cfg, int device, ozl_env** out);
int ozl_destroy(ozl_env* env);

/* Zero all private state (root = initial pose, thrust 0, target (0,0,1)), reset the step counter and
 * the metrics, and set the RNG seed.  The caller re-initialises its own reset_buf (=1) / progress_buf (=0)
 * as VecTask.allocate_buffers does (tasks/base/vec_task.py:254-277). */
int ozl_reset_all(ozl_env* env, uint64_t seed, void* stream);

/* One fused env step == VecTask.step (tasks/base/vec_task.py:313-359) with Ouzelum's hooks
 * (tasks/ouzelum.py:218-295) and gym.simulate replaced by the in-kernel rigid-body integrator.
 *   actions  [N,4] f32 in    (clamped to +-clip_actions inside)
 *   obs      [N,13] f32 out  (already clamped to +-clip_obs, i.e. obs_dict["obs"])
 *   rew      [N] f32 out
 *   reset    [N] i64 in/out  (reset_buf: request from the previous step in, new flag out)
 *   progress [N] i64 in/out  (progress_buf)
 *   timeout  [N] u8 out      (timeout_buf as bool; may be NULL)
 *   ep_ret   [N] f32 out     (episode return at episode end, RecordEpisodeStatisticsTorch "r"; may be NULL) */
int ozl_step(ozl_env* env, const float* actions, float* obs, float* rew, int64_t* reset, int64_t* progress,
             uint8_t* timeout, float* ep_ret, void* stream);

/* Zero-copy variant for a HOST consumer: `actions_host`, `obs_host`, `rew_host`, `done_host` are page-locked host buffers
 * mapped into the device address space (cudaHostAlloc / torch pinned memory: under UVA the host pointer IS the device
 * pointer).  The kernel reads the actions and writes observation, reward and a compact done flag (u8) straight across
 * PCIe, so one control step is one launch + one stream synchronise -- no separate H2D/D2H copies.  reset / progress stay
 * in device memory.  Replaces the `.to(rl_device)` copies of VecTask.step (vec_task.py:353-359) when rl_device is the CPU. */
int ozl_step_host(ozl_env* env, const float* actions_host, float* obs_host, float* rew_host, uint8_t* done_host,
                  int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream);

/* ozl_step_host + cudaStreamSynchronize in one call, arguments in a block the caller can fill once: the per-step cost on the
 * host side is one foreign call.  When it returns 0 the host buffers hold this step's results. */
typedef struct ozl_host_io {
    const float* actions_host;  /* [N,4] pinned */
    float* obs_host;            /* [N,13] pinned */
    float* rew_host;            /* [N] pinned */
    uint8_t* done_host;         /* [N] pinned */
    int64_t* reset_host;        /* [N] pinned or NULL: reset_buf mirrored with the reference's dtype (vec_task.py:353-359) */
    int64_t* reset;             /* [N] device */
    int64_t* progress;          /* [N] device */
    uint8_t* timeout;           /* [N] device or NULL */
    float* ep_ret;              /* [N] device or NULL */
} ozl_host_io;
int ozl_step_host_sync(ozl_env* env, const ozl_host_io* io, void* stream);
/* The two halves of ozl_step_host_sync, for a host consumer that pipelines several handles on several streams: launch only, and
 * a bare cudaStreamSynchronize (so that a binding needs no CUDA runtime of its own). */
int ozl_step_host_launch(ozl_env* env, const ozl_host_io* io, void* stream);
int ozl_stream_sync(void* stream);
/* Completion of the last ozl_step_host* launch of `env`: polls the completion word the step kernel's last block writes to pinned
 * host memory after all its result stores (a stream synchronise costs ~6 us more per step); falls back to synchronising
 * `stream` if the word does not arrive (which also reports CUDA errors).  ozl_step_host_sync = launch + this. */
int ozl_step_host_wait(ozl_env* env, void* stream);

/* Same step with the target supplied by the caller every step instead of being re-sampled in-kernel: the landing
 * family, whose target rides on a ground vehicle (tasks/landing.py:373-374, lando.py, landed.py).  target3 [N,3] f32. */
int ozl_step_tracking(ozl_env* env, const float* actions, const float* target3, float* obs, float* rew,
                      int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream);

/* Same step actuated by a body wrench instead of rotor thrust-rate commands: wrench4 [N,4] f32 = (fz, tx, ty, tz) on
 * the base link in LOCAL_SPACE, as the classical-control tasks apply it (tasks/lee_landed.py:316-330,
 * tasks/ekf_lee_landed.py:504-530).  No action clamp; target3 may be NULL (use the stored target). */
int ozl_step_wrench(ozl_env* env, const float* wrench4, const float* target3, float* obs, float* rew,
                    int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream);

/* Apply pending resets to the private state WITHOUT stepping: for envs with reset != 0 the spawn pose / target / fault
 * schedule / randomised parameters are drawn exactly as the next ozl_step* will draw them again (the draws are pure
 * functions of (seed, env, step counter), so re-applying is idempotent).  reset / progress buffers, metrics and the step
 * counter are untouched.  Lets composite tasks see the post-reset state in their pre-physics code, as the reference does
 * (reset_idx runs first in pre_physics_step, tasks/ekf_lee_landed.py:312-314, lee_landed.py:267-270). */
int ozl_apply_resets(ozl_env* env, const int64_t* reset, void* stream);

/* Privileged critic state (asymmetric actor-critic: the reference's numStates / states_buf / obs_dict["states"],
 * tasks/base/vec_task.py:104,121-122,145-151).  OZL_STATES_WIDTH float32 per env, row-major [N, OZL_STATES_WIDTH], written by
 * the same launch as the observation, from the same post-step registers (an env flagged for reset shows its terminal state).
 * Every slot is clamped to +-clip_obs like the observation.
 *   OZL_STATE_OBS .. +12        the CLEAN observation: before the sensor-fault model (pomdp_mode), after the clamp
 *   OZL_STATE_THRUST .. +3      rotor thrust state T0..T3 / thrust_max
 *   OZL_STATE_EFF .. +3         per-rotor effectiveness applied this step: 1, except the faulted rotor's effectiveness while its
 *                               fault is active (all 1 on wrench-actuated steps)
 *   OZL_STATE_MASS .. _ARM      per-env mass, ixx, iyy, izz, arm / their ozl_cfg values (exactly 1 when not randomised)
 *   OZL_STATE_THRUST_SCALE      per-env thrust scale (nominal 1)
 *   OZL_STATE_YAW_KM            per-env yaw_km (raw: its nominal may be 0)
 *   OZL_STATE_PROGRESS          progress after this step / max_episode_length
 *   OZL_STATE_POS .. +2         absolute root position / 3 (the observation's scaling; z is the die_z criterion)
 * Divisions are IEEE float32 divisions; the CPU reference (tests/states_ref.py, on the oracle's state) reproduces the row bit for bit. */
enum { OZL_STATE_OBS = 0, OZL_STATE_THRUST = 13, OZL_STATE_EFF = 17, OZL_STATE_MASS = 21, OZL_STATE_IXX = 22, OZL_STATE_IYY = 23,
       OZL_STATE_IZZ = 24, OZL_STATE_ARM = 25, OZL_STATE_THRUST_SCALE = 26, OZL_STATE_YAW_KM = 27, OZL_STATE_PROGRESS = 28,
       OZL_STATE_POS = 29, OZL_STATES_WIDTH = 32 };

/* Register a caller-owned [N, OZL_STATES_WIDTH] f32 buffer (16-byte aligned; any device-writable pointer) that every later
 * launch of ozl_step, ozl_step_tracking, ozl_step_wrench, ozl_step_host*, ozl_landing_step and ozl_lee_landed_step fills with
 * the privileged state above.  states = NULL unregisters (the steps then run the kernels without the output).
 * `width` must be OZL_STATES_WIDTH.  A captured CUDA graph keeps the buffer that was registered when it was captured.
 * While a buffer is registered, ozl_rollout and ozl_ekf_lee_landed_step refuse to run (non-zero return, ozl_last_error()):
 * their kernels do not write the state. */
int ozl_set_states_output(ozl_env* env, float* states, int32_t width);

/* Scenario table: per-env episode conditions that every reset of the env applies in place of the random draws, so that the
 * conditions of an episode no longer depend on the step at which the previous one ended (i.e. on the policy).  One float32 row
 * of OZL_SCENARIO_WIDTH per local env, row-major [N, OZL_SCENARIO_WIDTH]:
 *   OZL_SCN_POS .. +2          root position (absolute)                                      group "position"
 *   OZL_SCN_QUAT .. +3         attitude quaternion xyzw, unit                                group "attitude"
 *   OZL_SCN_LINVEL .. +2       linear velocity (world)                                       group "linear velocity"
 *   OZL_SCN_ANGVEL .. +2       angular velocity (world)                                      group "angular velocity"
 *   OZL_SCN_TARGET .. +2       target                                                        group "target"
 *   OZL_SCN_FAULT_ROTOR, _ONSET, _EFF   faulted rotor (0..3, or -1: no fault this episode), onset (progress step, an integer
 *                              in [0, 2^24)), effectiveness in [0, 1]                        group "fault"
 *   OZL_SCN_MASS .. _YAW_KM    mass, ixx, iyy, izz, arm, thrust_scale, yaw_km (absolute values, as params8 of ozl_set_params),
 *                              one group each
 *   OZL_SCN_RFAULT_ONSET, OZL_SCN_RFAULT_EFF .. +3   fault_mode 2 only: onset (an integer in [0, 2^24)) and e_0..e_3, each in
 *                              [0, 1]; four 1s mean no fault in that episode                 group "rotor faults"
 *   OZL_SCN_RESERVED .. 31     must be NaN (under fault_mode 2: slot 31 only, slots 26-30 are the rotor-faults group)
 * Slots 0-12 are laid out as root13 of ozl_set_state.  A group is either all NaN -- the env gets exactly what it gets without a
 * table: the draw, identity / zero for attitude and velocities, an unchanged value for a body parameter that is not randomised --
 * or all set, and then its values are used at every reset of the env.  An all-NaN table therefore gives results bit-identical to
 * no table.  A set target also holds through the periodic re-samples of the episode (target_period).  Not pinned by a table:
 * the per-step sensor-fault draws (flicker / noise), the observation and action noise lambdas, and the ground vehicle's
 * trajectory draws of the landing family.
 * The rows apply at the resets of ozl_step, ozl_step_tracking, ozl_step_wrench, ozl_step_host*, ozl_landing_step,
 * ozl_lee_landed_step and ozl_apply_resets; the landed flag and the episode bookkeeping are unchanged. */
enum { OZL_SCN_POS = 0, OZL_SCN_QUAT = 3, OZL_SCN_LINVEL = 7, OZL_SCN_ANGVEL = 10, OZL_SCN_TARGET = 13, OZL_SCN_FAULT_ROTOR = 16,
       OZL_SCN_FAULT_ONSET = 17, OZL_SCN_FAULT_EFF = 18, OZL_SCN_MASS = 19, OZL_SCN_IXX = 20, OZL_SCN_IYY = 21, OZL_SCN_IZZ = 22,
       OZL_SCN_ARM = 23, OZL_SCN_THRUST_SCALE = 24, OZL_SCN_YAW_KM = 25, OZL_SCN_RESERVED = 26, OZL_SCN_RFAULT_ONSET = 26,
       OZL_SCN_RFAULT_EFF = 27, OZL_SCENARIO_WIDTH = 32 };

/* Register the scenario table: `rows_host` is HOST memory, [N, OZL_SCENARIO_WIDTH] f32; `width` must be OZL_SCENARIO_WIDTH.
 * Every row is validated first and nothing is registered if one fails: reserved slots NaN; each group all NaN or all finite;
 * |x^2 + y^2 + z^2 + w^2 - 1| <= 1e-6 for the quaternion (the integrator keeps a unit quaternion unit with one Newton step and
 * needs a unit input); no target group when cfg.target_fixed is set (the target is driven by a vehicle or the caller); no fault
 * group unless cfg.fault_mode is 1 (under mode 2 the rotor-faults group instead, with the rules above); rotor in {-1, 0, 1, 2, 3},
 * onset an integer in [0, 2^24), effectiveness in [0, 1]; mass
 * and inertias in (1e-30, 1e30) (the step's reciprocals need positive normal floats), arm > 0, thrust_scale >= 0, yaw_km finite.
 * The rows are copied (stream-ordered on `stream`, which is then synchronised) into a device buffer the handle allocates on the
 * first registration and frees in ozl_destroy.  A later call overwrites the contents at the same address, so a CUDA graph
 * captured while a table is registered applies the new rows at its next resets.  rows_host = NULL unregisters.  Registering or
 * unregistering after a capture is not seen by that graph (it keeps the kernels it captured), as for ozl_set_states_output.
 * While a table is registered, ozl_rollout and ozl_ekf_lee_landed_step refuse to run (non-zero return, ozl_last_error()). */
int ozl_set_scenarios(ozl_env* env, const float* rows_host, int32_t width, void* stream);

/* Episode log: the step kernels append one record per episode that ends (reset flag raised) to a caller-owned buffer, with its
 * termination cause and its conditions, so that survival can be studied as a function of the fault and body parameters of each
 * episode -- which the next reset overwrites in the env's state.  A record is OZL_EPLOG_WIDTH four-byte slots (128 bytes), every
 * value from the registers of the step that ended the episode, after the step (the state an OZL_STATE_* row shows for an env
 * flagged for reset):
 *   OZL_EPLOG_ENV              global env id (env_id_base + local index), uint32 bits
 *   OZL_EPLOG_LENGTH           episode length: progress written by that step, int32 bits
 *   OZL_EPLOG_STEP .. +1       step index of that step (the RNG's time axis), uint64, low word first
 *   OZL_EPLOG_RETURN           episode return (the ep_ret output of that step)
 *   OZL_EPLOG_FLAGS            uint32: bit 0 time-out, bit 1 dist > die_dist, bit 2 z < die_z, bit 3 the env landed in this
 *                              episode (landed flag; metrics slot 2 counts it at the next step's reset), bit 4 rotor fault active
 *                              in that step (metrics slot 14)
 *   OZL_EPLOG_ONSET            fault onset (progress step), int32 bits; -1 when the episode had no fault scheduled
 *   OZL_EPLOG_DIST             final distance to the target, the float32 that was compared with die_dist
 *   OZL_EPLOG_EFF .. +3        per-rotor effectiveness of the episode: fault_mode 2 e_0..e_3 as drawn (not ramped); fault_mode 1
 *                              1 except the faulted rotor's effectiveness; no fault scheduled: all 1
 *   OZL_EPLOG_MASS .. _YAW_KM  mass, ixx, iyy, izz, arm, thrust_scale, yaw_km (absolute, the order of OZL_SCN_MASS ..)
 *   OZL_EPLOG_POS .. +2        final root position
 *   OZL_EPLOG_LINVEL .. +2     final linear velocity (world)
 *   OZL_EPLOG_TARGET .. +2     target of that step
 *   OZL_EPLOG_RESERVED .. 31   written 0
 * The contents of a record are deterministic (every draw is keyed by global env id and step: the same bits on every kernel and
 * sharding); the ORDER of the records is not. */
enum { OZL_EPLOG_ENV = 0, OZL_EPLOG_LENGTH = 1, OZL_EPLOG_STEP = 2, OZL_EPLOG_RETURN = 4, OZL_EPLOG_FLAGS = 5, OZL_EPLOG_ONSET = 6,
       OZL_EPLOG_DIST = 7, OZL_EPLOG_EFF = 8, OZL_EPLOG_MASS = 12, OZL_EPLOG_IXX = 13, OZL_EPLOG_IYY = 14, OZL_EPLOG_IZZ = 15,
       OZL_EPLOG_ARM = 16, OZL_EPLOG_THRUST_SCALE = 17, OZL_EPLOG_YAW_KM = 18, OZL_EPLOG_POS = 19, OZL_EPLOG_LINVEL = 22,
       OZL_EPLOG_TARGET = 25, OZL_EPLOG_RESERVED = 28, OZL_EPLOG_WIDTH = 32 };

/* Register the episode log: `records` is caller-owned device memory [capacity, OZL_EPLOG_WIDTH] f32 (16-byte aligned), `head` one
 * device uint64 the caller zeroes.  Every later launch of ozl_step, ozl_step_tracking, ozl_step_wrench, ozl_step_host*,
 * ozl_landing_step and ozl_lee_landed_step adds the records of the episodes it ends to *head atomically; record k (in the order
 * the additions hand them out) goes to row k if k < capacity and is dropped otherwise, but still counted: min(*head, capacity)
 * rows are valid, *head - capacity records were dropped.  Clearing the log is the caller's stream-ordered zeroing of *head, so
 * step, read and clear can all sit in one CUDA graph.  records = NULL unregisters (the steps then run the kernels without the
 * log).  Refused: env NULL, width != OZL_EPLOG_WIDTH, capacity < 1, misaligned records, head NULL.  A captured CUDA graph keeps
 * the log that was registered when it was captured.  While a log is registered, ozl_rollout and ozl_ekf_lee_landed_step refuse
 * to run (their kernels write no records); ozl_apply_resets ends no episode and writes none. */
int ozl_set_episode_log(ozl_env* env, float* records, int64_t capacity, uint64_t* head, int32_t width);

/* Mode-B throughput entry: K steps in ONE launch, state held in registers, actions a = 2u-1 drawn
 * in-kernel from the counter RNG; obs/rew are written for the LAST step only, reset/progress are
 * carried.  No reference counterpart (SURVEY 8d "mode B"). */
int ozl_rollout(ozl_env* env, int32_t K, float* obs, float* rew, int64_t* reset, int64_t* progress, void* stream);

/* State access (row-major AoS device buffers; any pointer may be NULL = skip).
 * Replaces the aliasing views root_states/thrusts/target_root_positions (tasks/ouzelum.py:67-96). */
int ozl_get_state(ozl_env* env, float* root13, float* thrust4, float* target3, float* ep_ret, void* stream);
int ozl_set_state(ozl_env* env, const float* root13, const float* thrust4, const float* target3,
                  const float* ep_ret, void* stream);
/* per-env parameters: params8 [N,8] = mass, ixx, iyy, izz, arm, thrust_scale, fault_effectiveness, yaw_km;
 * fault2 [N,2] i32 = fault rotor id, fault onset step (0x1FFFFFFF: never), landed flag in bit 31 of the onset word.
 * Mass and inertia must be positive normal floats (the step evaluates their IEEE reciprocals on a range-checked fast path). */
int ozl_get_params(ozl_env* env, float* params8, int32_t* fault2, void* stream);
int ozl_set_params(ozl_env* env, const float* params8, const int32_t* fault2, void* stream);
/* fault_mode 2: the per-rotor effectiveness e_0..e_3 of every env's current episode, eff4 [N,4] f32 device buffers (16-byte
 * aligned).  Stream-ordered copies, CUDA-graph capturable.  Non-zero return unless cfg.fault_mode == 2. */
int ozl_get_rotor_eff(ozl_env* env, float* eff4, void* stream);
int ozl_set_rotor_eff(ozl_env* env, const float* eff4, void* stream);

/* Step counter (the RNG's time axis): number of ozl_step's since ozl_reset_all.  Host-synchronising. */
int ozl_get_step_count(ozl_env* env, uint64_t* out, void* stream);
int ozl_set_step_count(ozl_env* env, uint64_t value, void* stream);

/* Metrics vector accumulated since the last clearing read (16 doubles, device pointer `out16`):
 *  [0] sum reward  [1] sum episode return of finished episodes  [2] episodes that ended after a landing  [3..7] reserved
 *  [8] env-steps  [9] finished episodes  [10] sum of finished episode lengths  [11] time-outs
 *  [12] dist>die_dist  [13] z<die_z  [14] env-steps with an active rotor fault  [15] resets applied
 * Every step path fills every slot the same way: ozl_rollout(K) adds what K single steps add, landed episodes included.
 * Replaces RecordEpisodeStatisticsTorch + the trainer's Python scan (RPO-LSTM/utils.py:20-35, main.py:105-113). */
int ozl_metrics_read(ozl_env* env, double* out16, int32_t clear, void* stream);

/* Multi-GPU sum of the metrics vector over NVLink peer memory (one process per GPU; csrc/peer_metrics.cu).  The only collective
 * on the path (SURVEY 8e); replaces an NCCL all-reduce of 128 bytes -- and the reference's host-side scan of `infos`
 * (RPO-LSTM/main.py:105-113) -- with 16-byte self-validating stores into every peer's mailbox, issued by the kernel that reads
 * the metrics: no collective kernel, no side stream, CUDA-graph capturable (no host-changing argument).
 *   create            one mailbox per rank (device memory of `device`)
 *   ipc_handle        64-byte cudaIpcMemHandle_t of the local mailbox, to be all-gathered by the caller (torch.distributed ...)
 *   connect_ipc       handles of ALL ranks, rank-major (world x 64 bytes); maps the peers' mailboxes
 *   connect_ptrs      same-process alternative: mailbox pointers (ozl_metrics_xchg_box) and device ordinals of all ranks; enables
 *                     peer access
 *   ozl_metrics_push  ozl_metrics_read + store this rank's 16 values into every rank's mailbox; `local16` (optional) receives this
 *                     rank's own values; if `prev_sum16` is given and an earlier exchange has not been summed yet, its sum is
 *                     written there first (one launch per exchange in steady state)
 *   ozl_metrics_sum   sum of the oldest exchange not summed yet, in rank order (bit-identical on every rank) -> sum16; waits for the
 *                     peers' stores (bounded: 10 s, then NaN and status.error = 1); no-op when nothing is outstanding
 * A rank may push at most 7 exchanges ahead of the slowest rank's sum. */
typedef struct ozl_metrics_xchg ozl_metrics_xchg;
int ozl_metrics_xchg_create(int32_t rank, int32_t world, int32_t device, ozl_metrics_xchg** out);
int ozl_metrics_xchg_destroy(ozl_metrics_xchg* x);
int ozl_metrics_xchg_ipc_handle(ozl_metrics_xchg* x, void* handle64);
int ozl_metrics_xchg_connect_ipc(ozl_metrics_xchg* x, const void* handles64xWorld);
int ozl_metrics_xchg_box(ozl_metrics_xchg* x, void** out);
int ozl_metrics_xchg_connect_ptrs(ozl_metrics_xchg* x, void* const* boxes, const int32_t* devices);
int ozl_metrics_push(ozl_env* env, ozl_metrics_xchg* x, double* local16, double* prev_sum16, int32_t clear, void* stream);
int ozl_metrics_sum(ozl_env* env, ozl_metrics_xchg* x, double* sum16, void* stream);
int ozl_metrics_xchg_status(ozl_metrics_xchg* x, uint64_t* pushed, uint64_t* summed, uint64_t* error, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Companion kernels.  All buffers are caller-owned device memory; `n` = number of envs.
 * ------------------------------------------------------------------------------------------------------------------ */

/* Lee geometric controllers.  Replaces Controller.__call__ (isaacgymenvs/controllers/controller.py:45-48) and
 * LeePositionController / LeeVelocityController / LeeAttitudeContoller.__call__
 * (controllers/position_control.py:19-109, velocity_control.py:17-112, attitude_control.py:17-78).
 *   mode 0 position, 1 velocity, 2 attitude (anything else: error "Invalid controller name", controller.py:34)
 *   state13 [n,13] f32 (pos, quat xyzw, linvel, angvel world), cmd4 [n,4] f32 (16-byte aligned)
 *   gains16  HOST pointer: kP[3], kV[3], kR[3], kOmega[3], scale_input[4]   (controllers/control_config.py:13-18)
 *   thrust [n] f32, torque3 [n,3] f32 ("m*g normalised thrust and inertia normalised torques") */
int ozl_lee_control(int32_t mode, int64_t n, const float* state13, const float* cmd4, const float* gains16,
                    float* thrust, float* torque3, void* stream);
/* Same controller, output packed as the body wrench the classical tasks apply: wrench4 [n,4] f32 =
 * (thrust_scale * thrust, tx, ty, tz) with thrust_scale = m g = 2 * 9.81 (tasks/lee_landed.py:296,313-314). */
int ozl_lee_wrench(int32_t mode, int64_t n, const float* state13, const float* cmd4, const float* gains16,
                   float thrust_scale, float* wrench4, void* stream);

/* Position/velocity/accel-bias Kalman filter bank.  State planes are SoA: x9xN = [9][n] f32, P81xN = [81][n] f32
 * (row-major 9x9 per env, full matrix -- the reference's (I-KH)P update is not symmetric in float32).
 * Replaces PVFilter.__init__ / prediction_step / correction_step (isaacgymenvs/PVFilter.py:7-110) and the per-env
 * Python loop around them (tasks/ekf_lee_landed.py:417-444). */
typedef struct ozl_pv_args {
    int64_t n;
    float* x9xN;
    float* P81xN;
    const float* accel3;      /* [n,3] body-frame specific force (prediction input)                    */
    const float* quat4;       /* [n,4] orientation, 16-byte aligned; xyzw if flip_qw else wxyz         */
    const float* pos_meas3;   /* [n,3] or NULL: position fix candidates                                */
    const float* vel_meas3;   /* [n,3] or NULL: velocity fix candidates                                */
    const uint8_t* pos_mask;  /* [n] or NULL: which envs take the position fix; NULL => trigger rule   */
    const uint8_t* vel_mask;  /* [n] or NULL                                                           */
    float dt;
    float acc_var[3];         /* process accel variance                                                */
    float pos_var[3];         /* used only if pos_var_given                                            */
    float vel_var[3];         /* used only if vel_var_given (the reference passes gps_var=None => R = 0, PVFilter.py:76-79) */
    int32_t pos_var_given, vel_var_given;
    int32_t flip_qw;          /* PVFilter.py:32-35                                                     */
    int32_t do_predict;       /* 0: corrections only                                                   */
    /* trigger rule when a mask is NULL: fix iff ((iter_base + env) % period) == phase; period 0 = never.
     * Reference (tasks/ekf_lee_landed.py:153-154,425-440, counters shared by all envs): position (7,6), velocity (3,0)
     * with iter_base = step * num_envs. */
    uint32_t pos_period, pos_phase, vel_period, vel_phase;
    uint64_t iter_base;
} ozl_pv_args;
int ozl_pv_init(int64_t n, float* x9xN, float* P81xN, void* stream);                       /* x = 0, P = 1000 I  (PVFilter.py:11-12) */
int ozl_pv_reset(int64_t n, float* x9xN, const int64_t* flags, const float* root13, void* stream);   /* x[flagged] = [pos, vel, 0]  (ekf_lee_landed.py:353-358); flags NULL = all */
int ozl_pv_step(const ozl_pv_args* args, void* stream);                                    /* predict, then gated position fix, then gated velocity fix: one launch */

/* Attitude EKF bank (float64).  q4xN = [4][n] f64 wxyz, P16xN = [16][n] f64.  Replaces EKF.__init__ / EKF.update
 * (isaacgymenvs/ahrs_ekf.py:982-1012, 1280-1337, `ang` branch) and the loop at tasks/ekf_lee_landed.py:378-391.
 * The a-priori quaternion is normalised inside (the reference's caller does q/|q|, ekf_lee_landed.py:386). */
int ozl_ekf_init(int64_t n, double* q4xN, double* P16xN, void* stream);                    /* q = (1,0,0,0), P = I4 (ahrs_ekf.py:995) */
int ozl_ekf_set_q(int64_t n, double* q4xN, const float* quat_xyzw, const int64_t* flags, void* stream);   /* Q_state[flagged] = quat[[3,0,1,2]]; flags NULL = all */
int ozl_ekf_update(int64_t n, double* q4xN, double* P16xN, const float* gyr3, const float* ang4, int32_t ang_xyzw,
                   double Dt, double g_noise, float* q_wxyz_f32_out /* [n,4] or NULL */, void* stream);

/* Glue kernels of EKFLeeLanded.pre_physics_step (isaacgymenvs/tasks/ekf_lee_landed.py:339-503).
 * ozl_sensor_frontend: sensors16 [n,16] = accel(3)|gyr(3)|ang xyzw(4)|pos(3)|vel(3) from the true root state, through the
 *   sensor-fault model when mode != 0 (:345-346,366-375,397-406); prev_linvel3 [n,3] is read then updated (:454).
 * ozl_waypoint_command: carrot-waypoint logic and controller-input assembly (:458-503): waypoint3 [n,3] in/out,
 *   est13 [n,13] = truth (warm-up) or [PV pos, true quat, PV vel, true angvel], cmd4 [n,4] = (waypoint, yaw 0). */
int ozl_sensor_frontend(int64_t n, const float* root13, float* prev_linvel3, float* sensors16, float dt, int32_t mode,
                        float pomdp_prob, uint64_t seed, uint64_t step, int64_t env_id_base, void* stream);
int ozl_waypoint_command(int64_t n, const float* root13, const float* pv_x9xN, const float* target3, float* waypoint3,
                         int32_t warmup, float* est13, float* cmd4, void* stream);

/* The whole estimator + controller chain of EKFLeeLanded.pre_physics_step (isaacgymenvs/tasks/ekf_lee_landed.py:308-530) as
 * ONE launch on the envs of `env`: reset handling, sensor front-end + sensor faults, attitude EKF, PV filter with the shared
 * trigger counters, carrot-waypoint logic, Lee position controller on the estimates, warm-up hover force.  The true root
 * state is read from the handle's private planes; the step index / warm-up flag come from the handle's device step counter
 * (CUDA-graph capturable).  Output: wrench4 [N,4] for ozl_step_wrench.  est13 / cmd4 are optional debug outputs (NULL ok). */
typedef struct ozl_ekf_lee_args {
    double* ekf_q4xN;
    double* ekf_P16xN;
    float* pv_x9xN;
    float* pv_P81xN;
    float* prev_linvel3;      /* [N,3] in/out   ekf_lee_landed.py:95,454 */
    float* waypoint3;         /* [N,3] in/out   :160,461-486             */
    const float* target3;     /* [N,3]          target riding on the vehicle */
    const int64_t* reset;     /* [N]            reset_buf                */
    float* wrench4;           /* [N,4] out      (m g thrust, torque) or the warm-up hover force */
    float* est13;             /* [N,13] out or NULL */
    float* cmd4;              /* [N,4] out or NULL  */
    const float* gains16;     /* HOST: kP, kV, kR, kOmega, scale_input   */
    float dt;
    float mg;                 /* 2 * 9.81       :459                     */
    float hover_force;        /* 2.09 * 9.81    :527                     */
    int64_t convergence_steps;/* ConvergenceTime :339                    */
    int32_t pomdp_mode;
    float pomdp_prob;
    uint32_t pos_period, pos_phase, vel_period, vel_phase;   /* (7,6,3,0) for 20 / 75 Hz at dt 0.01 */
    int32_t per_env_triggers; /* 0: the reference's counters shared by all envs; 1: every env counts its own steps */
    int64_t num_envs_total;   /* envs of the WHOLE job (all ranks); 0 = this handle's.  The shared counters advance once per
                                 env-iteration, so fix k of env e at step t is t * num_envs_total + global id(e): invariant to sharding */
    float acc_var[3], pos_var[3];
    double ekf_Dt, ekf_g_noise;
} ozl_ekf_lee_args;
int ozl_ekf_lee_step(ozl_env* env, const ozl_ekf_lee_args* args, void* stream);

/* The WHOLE EKFLeeLanded control step in one launch: vehicle carrying the target (ozl_husky_step), estimator + controller
 * (ozl_ekf_lee_step) and the physics / observation / reward / reset step with that wrench and target (ozl_step_wrench),
 * per env in one thread, state read once.  Replaces VecTask.step for isaacgymenvs/tasks/ekf_lee_landed.py
 * (pre_physics_step :308-530, post_physics_step :620-665).  `husky` follows the env's device step counter (its `step` /
 * `step_ptr` fields are ignored); `reset` must be the buffer named in `args->reset` (and `husky->reset` if set).
 * Float results agree with the three-launch sequence to rounding (this translation unit keeps FMA contraction on). */
struct ozl_husky_args;
int ozl_ekf_lee_landed_step(ozl_env* env, const ozl_ekf_lee_args* args, const struct ozl_husky_args* husky, float* obs,
                            float* rew, int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream);

/* Device address of the handle's step counter, for kernels that must follow it without a host round trip.
 * The counter is a 16-byte record of two uint64 words: word0 = base | (shift << 58), word1 = units, and
 *     step = (word0 & (2^58 - 1)) + (word1 >> (word0 >> 58)).
 * (Every step launch retires 2^shift work units with fire-and-forget reductions -- no last-block election on the step
 * path; see ouzelum_b200/csrc/step_counter.cuh.)  Read both words with one 16-byte relaxed load; ozl_get_step_count does
 * the same on the host.  The library's own consumers (ozl_pomdp_observation_dev, ozl_husky_step, ozl_ekf_lee_step) take
 * this pointer. */
int ozl_step_counter_ptr(ozl_env* env, const uint64_t** out);

/* Sensor-fault model on an [n,d] f32 array.  Replaces POMDPWrapper.observation (isaacgymenvs/utils/POMDP.py:23-42).
 * mode: OZL_POMDP_FLICKER / _NOISE / _FLICKER_NOISE (anything else: the reference's ValueError text).
 * Draws are counter-based: (seed, global env id, step, stream_id) -- stream_id separates several uses in one step. */
int ozl_pomdp_observation(int64_t n, int32_t d, int32_t mode, float pomdp_prob, uint64_t seed, uint64_t step,
                          int64_t env_id_base, int32_t stream_id, const float* in, float* out, void* stream);
/* Same, with the call index read from a DEVICE counter (ozl_step_counter_ptr) -- no host-changing argument, so a whole
 * policy -> step -> sensor-fault iteration can sit in one CUDA graph. */
int ozl_pomdp_observation_dev(int64_t n, int32_t d, int32_t mode, float pomdp_prob, uint64_t seed, const uint64_t* step_ptr,
                              int64_t env_id_base, int32_t stream_id, const float* in, float* out, void* stream);

/* RecordEpisodeStatisticsTorch.step (isaacgymenvs/RPO-LSTM/utils.py:20-35) in one launch:
 * ep_ret += rew; ep_len += 1; ret_out = ep_ret; len_out = ep_len; ep_ret *= 1-done; ep_len *= 1-done. */
int ozl_episode_stats(int64_t n, const float* rew, const int64_t* done, float* ep_ret, int32_t* ep_len,
                      float* ret_out, int32_t* len_out, void* stream);

/* Waypoint-following ground vehicle that carries the landing target (kinematic differential drive).
 * Replaces Landing.set_husky_actions / reset_completed_trajectories (isaacgymenvs/tasks/landing.py:208-244,319-364),
 * differential_drive (utils/controllers.py:15-43) and the target-on-vehicle rule (landing.py:373-374).
 *   pose4 [n,4] f32 = x, y, heading, scale*direction      idx2 [n,2] i32 = trajectory id, waypoint index
 *   tables204x2 [204,2] f32 = lemniscate(4,100) | circle(2,100) | square(4,8)   (utils/trajectories.py, landing.py:108-112)
 *   reset [n] i64 or NULL: drone reset flags (a vehicle beyond respawn_limit is re-spawned, landing.py:263-270)
 *   wheels4 [n,4] f32 out or NULL (right,left,right,left), target3 [n,3] f32 out */
typedef struct ozl_husky_args {
    int64_t n;
    float* pose4;
    int32_t* idx2;
    const float* tables204x2;
    const int64_t* reset;
    float* wheels4;
    float* target3;
    uint64_t seed, step;
    const uint64_t* step_ptr; /* if non-NULL the step index is read from this DEVICE address instead of `step` */
    int64_t env_id_base;
    float dt;             /* 0.01                                      */
    float dist_thresh;    /* 0.2        landing.py:319                 */
    float kp_lin, kp_ang; /* 3.0, 1000  landing.py:362                 */
    float ang_thresh;     /* 0.005      utils/controllers.py:16        */
    float x_offset;       /* +0.08 (landing.py:374) / -0.08 (ekf_lee_landed.py:629) */
    float target_z;       /* 0.377      landing.py:76                  */
    float respawn_limit;  /* 2 * envSpacing  landing.py:266-267        */
} ozl_husky_args;
int ozl_husky_init(const ozl_husky_args* args, void* stream);
int ozl_husky_step(const ozl_husky_args* args, void* stream);

/* Landing / Landed in ONE launch: the vehicle step (ozl_husky_step) and the tracking step (ozl_step_tracking) per env in one
 * thread.  Replaces VecTask.step for isaacgymenvs/tasks/landing.py (set_husky_actions :319-364, target rule :373-374,
 * pre/post_physics_step) and landed.py.  `husky` follows the handle's device step counter (`step` / `step_ptr` ignored). */
int ozl_landing_step(ozl_env* env, const float* actions, const ozl_husky_args* husky, float* obs, float* rew, int64_t* reset,
                     int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream);

/* LeeLanded in ONE launch (isaacgymenvs/tasks/lee_landed.py:263-330): vehicle, Lee position controller on the true state after
 * reset_idx towards the fixed command `cmd` (:299-302, (0,0,1,yaw 0)), wrench = (mg * thrust, torque) on the base link (:313-314),
 * landing detector on the CONTROLLER target within cfg.land_cutoff (:305,318-322), physics / observation / reward / reset. */
typedef struct ozl_lee_landed_args {
    const float* gains16;     /* HOST: kP, kV, kR, kOmega, scale_input   (controllers/control_config.py:13-18) */
    float cmd[4];             /* controller target x, y, z, yaw */
    float mg;                 /* 2 * 9.81   lee_landed.py:296 */
    float* wrench4;           /* [N,4] out or NULL: the wrench the controller asked for (before the landing / reset zeroing) */
} ozl_lee_landed_args;
int ozl_lee_landed_step(ozl_env* env, const ozl_lee_landed_args* args, const ozl_husky_args* husky, float* obs, float* rew,
                        int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream);

/* Stock Quadcopter hover task (BASELINE config 1): one fused step.  Replaces VecTask.step with the hooks of
 * isaacgymenvs/tasks/quadcopter.py:280-330,359-418.  All state is caller-owned AoS device memory:
 *   actions12 [n,12] in; root13 [n,13], dof_pos8 [n,8], dof_target8 [n,8], thrust4 [n,4] in/out;
 *   obs21 [n,21], rew [n] out; reset [n] i64, progress [n] i64 in/out; timeout [n] u8 out or NULL.
 * `step` is the caller-maintained step index (the RNG's time axis).  mass / inertia: the composite rigid body of the
 * procedurally built vehicle (quadcopter.py:121-202), computed by the host binding. */
typedef struct ozl_quadcopter_args {
    int64_t n;
    const float* actions12;
    float* root13;
    float* dof_pos8;
    float* dof_target8;
    float* thrust4;
    float* obs21;
    float* rew;
    int64_t* reset;
    int64_t* progress;
    uint8_t* timeout;
    uint64_t seed, step;
    int64_t env_id_base;
    int32_t max_episode_length;   /* 500   cfg/task/Quadcopter.yaml:10 */
    int32_t substeps;             /* 2                                 */
    float dt, gravity_z, clip_actions, clip_obs;
    float mass, ixx, iyy, izz;
    uint64_t* step_record;        /* optional: DEVICE step-counter record (ozl_step_record_init).  When set, the kernel takes the
                                     step index from it and advances it itself -- no host-changing argument, so the launch can be
                                     captured in a CUDA graph -- and `step` is ignored */
} ozl_quadcopter_args;
int ozl_quadcopter_step(const ozl_quadcopter_args* args, void* stream);

/* Observation / action noise of the reference's domain randomisation (the `noise_lambda`s of tasks/base/vec_task.py:576-646),
 * applied in place to an [n,width] f32 tensor:
 *     gaussian  out = op(x, (corr * b_corr + a_corr) + randn * b + a)        a = mu,  b = var  (used as the std factor, as there)
 *     uniform   out = op(x, (corr * (b_corr - a_corr) + a_corr) + rand * (b - a) + a)       a = lo,  b = hi
 * op = + (additive) or * (scaling); `corr` is a standard normal drawn once per randomisation event (`corr_epoch`) and kept until the
 * next one, randn / rand are fresh every `step`.  The schedule (linear / constant) is applied by the caller when the event happens
 * (ouzelum_b200.vec_task.VecTask.apply_randomizations).  `step_ptr` (optional): a device step-counter record; the kernel then
 * uses its value + `step_offset` instead of `step` (CUDA-graph capturable).  `clip` > 0 clamps the result to [-clip, clip].
 * `which`: 0 observations, 1 actions (separate random streams). */
typedef struct ozl_noise_lambda {
    int32_t distribution;         /* OZL_DR_GAUSSIAN or OZL_DR_UNIFORM */
    int32_t operation;            /* OZL_DR_ADDITIVE or OZL_DR_SCALING */
    float a, b, a_corr, b_corr;
} ozl_noise_lambda;
int ozl_noise_lambda_apply(int64_t n, int32_t width, float* tensor, const ozl_noise_lambda* spec, float clip, uint64_t seed,
                           uint64_t step, const uint64_t* step_ptr, int64_t step_offset, uint64_t corr_epoch, int64_t env_id_base,
                           int32_t which, void* stream);

/* A stand-alone device step counter for kernels without an env handle: 16 bytes of caller-owned device memory (16-byte aligned),
 * the same record ozl_step_counter_ptr describes.  `n_envs` fixes how many 128-env blocks retire a work unit per step. */
int ozl_step_record_init(uint64_t* record_dev, int64_t n_envs, uint64_t step, void* stream);
int ozl_step_record_read(const uint64_t* record_dev, uint64_t* out, void* stream);   /* synchronises the stream */

const char* ozl_last_error(void);
int ozl_abi_version(void);
int ozl_cfg_size(void);            /* sizeof(ozl_cfg): lets a binding verify its struct mirror */

#ifdef __cplusplus
}
#endif
#endif /* OUZELUM_B200_H */
