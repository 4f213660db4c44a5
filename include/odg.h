/* odg.h — C ABI of libodgsim: the B200-native batched replacement for the OpenDOG hot path.
 *
 * The reference has no FFI for this path: it calls the `mujoco` Python bindings and its own numpy
 * reward code once per environment per step. Each entry point below replaces, for a whole batch of
 * environments resident in HBM, the reference interface cited next to it (paths relative to
 * /root/reference/Code/mujoco). INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions: plain pointers and sizes only; every `*_dev` pointer is caller-owned device memory
 * on the handle's device (e.g. `tensor.data_ptr()`), row-major [num_envs][dim] unless stated;
 * calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream);
 * a handle is bound to one device and is not re-entrant; distinct handles are independent (one per
 * rank). Return value: 0 on success, negative OdgStatus otherwise; never throws, never exits.
 * Per-environment physics failure (non-finite state) is not an error: it surfaces as
 * terminated=1, mirroring `is_healthy` (rewards/walk_environment_reward_calc.py:117-121) and the
 * `except mujoco.FatalError` path (sim2real/train.py:282-283).
 */
#ifndef ODG_H
#define ODG_H

#include <stddef.h>
#include <stdint.h>
#include "odg_model.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct OdgSim OdgSim;

enum OdgStatus {
  ODG_OK = 0,
  ODG_ERR_INVALID = -1,      /* bad argument / unsupported model */
  ODG_ERR_CUDA = -2,         /* CUDA runtime error (see odg_last_error) */
  ODG_ERR_NO_DEVICE = -3,    /* no CUDA device: there is NO CPU fallback */
  ODG_ERR_ALLOC = -4
};

enum OdgTask {
  ODG_TASK_WALK = 0,         /* ScaleActionWrapper(WalkEnvironmentV0): obs 33, act 8 */
  ODG_TASK_JUMP = 1          /* JumpEnvironmentV0 (environments/JumpEnvironment.py:70-119 + rewards/jump_environment_reward_calc.py)
                                on the 12-actuator model: obs 21, act 12 = ctrl targets (use scale_actions = 0,
                                reset_noise_scale = 0.1 as the reference does) */
};

/* Environment configuration. Defaults (odg_default_config) are the reference's constants. */
typedef struct OdgEnvConfig {
  int task;                  /* OdgTask */
  int frame_skip;            /* mj_step calls per env step; WalkEnvironment.py:36 -> 10 */
  int max_episode_steps;     /* truncation; WalkEnvironment.py:52,63 -> 15.0/(0.002*10) = 750 */
  int auto_reset;            /* 1 = SB3 VecEnv worker semantics (train/train.py:81-86): done envs are
                                reset inside odg_step and the returned obs is the reset obs */
  int solver_iterations;     /* max Newton iterations per substep (MuJoCo default 100, tol 1e-8);
                                the kernel exits early on convergence (mean ~5). default 30 */
  int ls_iterations;         /* line-search passes per Newton iteration; each pass evaluates phi' at 4 step
                                lengths at once (first {0.25,0.5,1,2}, then a geometric ladder below the smallest step
                                tried while phi' is still negative there, else 4 interior points of the bracket). At least
                                3 (else ODG_ERR_INVALID): with 1 or 2 passes a step below 0.25 is not resolved and the solve
                                can stall at the iteration cap far from the optimum. default 4 */
  float solver_tolerance;    /* the Newton iteration stops after a full step whose inf-norm is <= tol * (1 + |qacc|_inf).
                                The result is NOT accurate to ~tol^2, and not always to tol * (1 + |qacc|_inf) either: the
                                step is computed with the iterate's active rows, and where the optimum has fewer active rows a
                                short step can stop up to ~55x that distance from it (rare; the states are pinned as expected
                                failures in tests/test_solver_optimality.py). default 1e-4 */
  float ls_tolerance;        /* a step length alpha is accepted without further refinement when
                                |phi'(alpha)| <= ls_tolerance * |phi'(0)|. It changes the path of the iteration and its
                                length: tests/test_solver_optimality.py checks ls_iterations in {3, 4, 8} x ls_tolerance in
                                {0.01, 0.1, 0.5} against the fp64 optimum; with 0.5 a state can need more than the
                                default 30 iterations. default 0.1 */
  float reset_noise_scale;   /* reward_calc:106 -> 0.02 */
  int scale_actions;         /* 1 = apply ScaleActionWrapper.action (ScaleActionEnvironment.py:21-23)
                                to actions in [-1,1]; 0 = actions are ctrl targets in rad */
  int launch_lanes;          /* launch shape of the step kernel (schedule only: never changes a result bit, tests pin that).
                                Active lanes per warp: 32, 16, 8 or 4 = 8, 4, 2 or 1 environments per warp; 0 = chosen from the
                                batch size (8 environments per warp unless the batch has fewer warps than the GPU has SMs) */
  int first_env_id;          /* global id of env 0 of this handle (rank * num_envs): RNG streams are
                                keyed by global env id so results do not depend on the sharding */
  int obs_layout;            /* 0 = WalkEnvironmentV0._get_obs (WalkEnvironment.py:115-136): 9 + 3*nu values
                                [2 v, 0.25 w, 2 v_des, q - key_ctrl[0,7:] (length-1 slice broadcast), 0.05 qd, last_action];
                                1 = the 12-actuator layout of landing_environment.py:116-136 plus the desired velocity
                                (the "48" of BASELINE configs[2]): 12 + 3*nu values
                                [2 v, 0.25 w, projected_gravity (reward_calc get_projected_gravity, its Euler-angle
                                formula), 2 v_des, q - key_qpos[0,7:], 0.05 qd, last_action] */
  int launch_block;          /* threads per block of the step kernel: 32, 64 or 128; 0 = 64 */
  int launch_lockstep;       /* 1 = the warps of a block take Newton iterations in lockstep (one barrier per iteration;
                                pays when the batch is several waves deep), 2 = pairs of warps inside 128-thread blocks do
                                (named barriers; needs launch_lanes 32 and launch_block 128 or 0), 0 = never, -1 = chosen
                                from the batch size */
  int launch_fat;            /* 1 = the instantiation of the step kernel that keeps per-contact Jacobian columns and line-search
                                coefficients in local memory instead of recomputing them, 0 = the lean one, -1 = chosen by the
                                library (the former at every batch size as of the end of round 2). Schedule only: results
                                are bit-identical */
} OdgEnvConfig;

/* Optional per-step outputs (any pointer may be NULL). WalkEnvironment.py:65-72 `info`. */
typedef struct OdgInfoPtrs {
  float* x_position;             /* [N] */
  float* y_position;             /* [N] */
  float* distance_from_origin;   /* [N] */
  float* paw_contact_forces;     /* [N][4][6], reward_calc:351-370 incl. its frame quirks */
  float* patterns_matches;       /* [N], second diagonal_gait_reward call */
  float* linear_vel_tracking_reward; /* [N] */
  float* reward_ctrl;            /* [N], sum(qfrc_actuator[-8:]^2) */
  float* terminal_obs;           /* [N][obs_dim]: obs before auto-reset (SB3 info["terminal_observation"]) */
  uint8_t* paws_in_ground;       /* [N][4] FL FR BL BR */
  int32_t* gait_reward;          /* [N] integer value of the first diagonal_gait_reward call */
  /* solver / parity diagnostics of the LAST substep's forward pass */
  float* qacc;                   /* [N][nv] MuJoCo dof order and frames */
  int32_t* ncon;                 /* [N] number of contacts */
  float* contact_normal_force;   /* [N] sum of contact normal forces */
  int32_t* solver_iters;         /* [N] Newton iterations used in the last substep */
  int32_t* ls_evals;             /* [N] line-search passes used in the last substep */
  float* reward_unclipped;       /* [N] rewards - costs BEFORE the max(0, .) clip of WalkEnvironment.py:84 (MPPI cost) */
  /* 12-actuator model only (NULL elsewhere) */
  float* cfrc_ext;               /* [N][13][6] data.cfrc_ext[1:] after do_simulation: per body [torque about the robot's
                                    centre of mass, force], world axes (jump_environment_reward_calc.py:131-133) */
  float* task_terms;             /* [N][10] jump task: compute_rewards' reward_info, weighted, in its key order */
} OdgInfoPtrs;

void odg_default_config(OdgEnvConfig* cfg);

/* Replaces `mujoco.MjModel.from_xml_path` + `mujoco.MjData` x num_envs + env construction
 * (WalkEnvironment.py:33-54, train/train.py:63-87). Uploads model constants, allocates the SoA
 * state, samples per-env desired velocities (reward_calc:75,301-305) and leaves every env at the
 * noise-free home keyframe; call odg_reset next. */
int odg_create(const OdgModel* model, const OdgEnvConfig* cfg, int num_envs, int device,
               uint64_t seed, OdgSim** out);
void odg_destroy(OdgSim* sim);

int odg_num_envs(const OdgSim* sim);
int odg_obs_dim(const OdgSim* sim);
int odg_act_dim(const OdgSim* sim);
int odg_nq(const OdgSim* sim);
int odg_nv(const OdgSim* sim);

/* Replaces `env.reset()` (MujocoEnv.reset -> mj_resetData -> WalkEnvironment.py:138-151).
 * mask_dev: [N] bytes, nonzero = reset that env; NULL = all. obs_dev: [N][obs_dim] or NULL. */
int odg_reset(OdgSim* sim, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* Replaces `env.step(action)` for all envs (WalkEnvironment.py:56-79: do_simulation = frame_skip x
 * mj_step, _get_obs, _calculate_rewards, is_healthy, truncation; ScaleActionEnvironment.py:21-23;
 * SB3 auto-reset when cfg.auto_reset). action_dev: [N][act_dim]. */
int odg_step(OdgSim* sim, const float* action_dev, float* obs_dev, float* reward_dev,
             uint8_t* terminated_dev, uint8_t* truncated_dev, const OdgInfoPtrs* info, void* stream);

/* `odg_step` for a caller whose policy lives on the HOST (stable-baselines3's numpy rollout loop, train/train.py:117-158;
 * the batch-1 loop of sim2real/train.py:537-549): ONE call = host actions in, host results out. Copies
 * action_host [N][act_dim] (any host memory; through action_pinned — a page-locked staging buffer of the same size, or
 * NULL when action_host is page-locked itself) to action_dev, takes the step into obs_dev / reward_dev / terminated_dev /
 * truncated_dev (+ info), copies `out_bytes` bytes from out_dev to out_host (page-locked; the caller lays its output
 * tensors out in one device slab so that one copy brings all of them), and waits for the stream: when it returns, out_host
 * holds the step's results. out_dev / out_host may be NULL (no copy back).
 * Zero-copy forms (page-locked memory has the same address on the device under unified addressing): pass the page-locked
 * source itself as action_dev and the kernel reads the actions in place over PCIe (no H2D copy is issued); pass
 * page-locked obs_dev / reward_dev / terminated_dev / truncated_dev with out_dev = out_host = NULL and the kernel writes
 * the results where the host reads them. Same results; saves the copy engine's launch latencies on small batches. */
int odg_step_host(OdgSim* sim, const float* action_host, float* action_pinned, float* action_dev,
                  float* obs_dev, float* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                  const OdgInfoPtrs* info, const void* out_dev, void* out_host, size_t out_bytes, void* stream);

/* Test hook: one `mj_forward` on the current state (no integration), then the same
 * obs/reward/termination code as odg_step, with `ctrl_dev` [N][act_dim] already in ctrl units.
 * Lets reward/done/reset logic be compared bit-for-bit on identical states. Never auto-resets. */
int odg_evaluate(OdgSim* sim, const float* ctrl_dev, float* obs_dev, float* reward_dev,
                 uint8_t* terminated_dev, uint8_t* truncated_dev, const OdgInfoPtrs* info, void* stream);

/* Replace reads/writes of `data.qpos` / `data.qvel` (parity tests: identical initial states).
 * qpos_dev [N][nq], qvel_dev [N][nv], MuJoCo layout. set_state also zeroes the solver warm start
 * (as mj_resetData does) unless qacc_warmstart_dev [N][nv] is given. */
int odg_get_state(OdgSim* sim, float* qpos_dev, float* qvel_dev, void* stream);
int odg_set_state(OdgSim* sim, const float* qpos_dev, const float* qvel_dev,
                  const float* qacc_warmstart_dev, void* stream);
/* Env-side state kept outside mjData by the reference (reward_calc:67-69,75,107; WalkEnvironment.py:53):
 * step counter [N] i32, gait index [N] i32, consecutive matches [N] i32, last action [N][act_dim],
 * desired velocity [N][3], last_action_is_reset [N] u8. NULL pointers are skipped. */
int odg_get_env_state(OdgSim* sim, int32_t* step, int32_t* gait_index, int32_t* gait_matches,
                      float* last_action, float* desired_velocity, uint8_t* fresh, void* stream);
int odg_set_env_state(OdgSim* sim, const int32_t* step, const int32_t* gait_index,
                      const int32_t* gait_matches, const float* last_action,
                      const float* desired_velocity, const uint8_t* fresh, void* stream);

/* Change the number of mj_step calls per odg_step (open-loop playback holds each target for duration / timestep
 * substeps: sim2real/run.py:286-330). */
int odg_set_frame_skip(OdgSim* sim, int frame_skip);

/* Number of kernels this library has launched on behalf of `sim` (bench.py's gpu_launches). */
long long odg_launch_count(const OdgSim* sim);

/* Thread-local description of the last error on this thread. */
const char* odg_last_error(void);
/* Library / build identification, e.g. "odgsim 0.1 sm_100a". */
const char* odg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ODG_H */
