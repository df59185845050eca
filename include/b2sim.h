/* b2sim.h — C ABI of the B200-native batched physics step (libb2sim.so).
 *
 * Drop-in boundary: these entry points are what mjlab's `Simulation` class
 * (reference src/mjlab/sim/sim.py:94-198) needs from its physics backend. In the reference
 * that backend is the Python package mujoco_warp, reached from four call sites:
 *   mjwarp.put_model  sim.py:110      -> b2_create (model upload)
 *   mjwarp.put_data   sim.py:113-119  -> b2_create (nworld / nconmax / njmax sizing, Data alloc)
 *   mjwarp.step       sim.py:136,195  -> b2_step / b2_step_n
 *   mjwarp.forward    sim.py:139,187  -> b2_forward
 * plus the zero-copy field access that WarpBridge/TorchArray provide (sim_data.py:15-229)
 *   getattr(wp_data, name) / wp.to_torch -> b2_get_field
 * and the per-world model tiling of sim/randomization.py:20-55
 *   expand_model_fields -> b2_expand_model_field.
 * No torch types cross this boundary: plain pointers, sizes and a CUDA stream handle.
 * All functions return 0 on success, non-zero on error (message via b2_last_error()).
 * Nothing in b2_step/b2_forward allocates, synchronises or touches the host: they only enqueue
 * kernels on the given stream and are CUDA-graph capturable.
 */
#ifndef B2SIM_H_
#define B2SIM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- model description handed in by the host (compiled by mjlab_b200.compiler) ---------- */
enum { B2_F64 = 0, B2_I32 = 1, B2_F32 = 2 };

typedef struct B2Array {
  const char* name; /* mjModel-style field name, e.g. "body_pos", "nq", "opt_timestep" */
  int32_t dtype;    /* B2_F64 or B2_I32 */
  int64_t n;        /* number of elements */
  const void* data; /* host pointer, valid during b2_create only */
} B2Array;

typedef struct B2ModelDesc {
  int32_t narray;
  const B2Array* arrays;
  double gravity[3];
} B2ModelDesc;

/* ---- tensor view returned for a Data / Model field ---------------------------------------- */
enum { B2_DATA = 0, B2_MODEL = 1 };

typedef struct B2Tensor {
  void* ptr;         /* device pointer */
  int32_t dtype;     /* B2_F32 or B2_I32 */
  int32_t ndim;      /* <= 4; shape[0] == nworld for Data and for expanded Model fields, else 1 */
  int64_t shape[4];
  int64_t stride[4]; /* in elements; rows are padded to 16 B so they can be bulk-copied (TMA) */
  int32_t device;    /* CUDA ordinal */
} B2Tensor;

typedef struct B2Stats {
  int32_t ncon_max, ncon_cap;   /* max contacts in any world / per-world capacity */
  int32_t nefc_max, nefc_cap;   /* max constraint rows in any world / njmax */
  int32_t overflow_worlds;      /* worlds that hit a capacity (contacts truncated, in pair order) */
  int32_t niter_max;            /* max Newton iterations used by any world in the last step */
  double ncon_mean, nefc_mean, niter_mean;
} B2Stats;

typedef struct b2_sim b2_sim;

/* Create a simulation: uploads the model, allocates Data for `nworld` worlds on `cuda_device`,
 * initialises qpos=qpos0 and runs one forward pass so every derived field is valid
 * (reference sim.py:106-107 relies on a forwarded MjData; SURVEY.md §8a S1b).
 *   ncon_per_world <= 0 : default capacity; njmax <= 0 : default.
 *   njmax is recorded (B2Stats.nefc_cap) but never truncates: the solver is matrix-free, so constraint rows
 *   need no storage and every contact within the contact capacity gets its rows (upstream drops rows past njmax). */
int b2_create(const B2ModelDesc* model, int nworld, int ncon_per_world, int njmax,
              int cuda_device, b2_sim** out);
int b2_destroy(b2_sim* sim);

/* Zero-copy view of a field. Pointers stay valid for the lifetime of the sim, except that
 * b2_expand_model_field re-points the named Model field.  The model-pointer table travels to the
 * kernels as a by-value launch parameter, so CUDA graphs captured before an expansion must be
 * re-captured (mjlab does: manager_based_rl_env.py:102-104; our Simulation does it lazily).
 * A Model view of body_pos, body_quat, jnt_pos, jnt_axis or qpos0 (from either call, at any nworld)
 * turns off the kinematic records cached from them at create time, which also changes that table. */
int b2_get_field(b2_sim* sim, int which, const char* name, B2Tensor* out);
int b2_num_fields(b2_sim* sim, int which);
const char* b2_field_name(b2_sim* sim, int which, int index);

/* Tile a Model field to a real leading nworld dimension (reference randomization.py:20-55). */
int b2_expand_model_field(b2_sim* sim, const char* name, void* cuda_stream, B2Tensor* out);

/* Options (set and get): "iterations", "ls_iterations", "tolerance", "ls_tolerance", "timestep",
 * "integrator", "solver" (1 CG, 2 Newton), "ls_parallel" (set only; accepted, the line search is exact),
 * "sorted_dispatch" (heavy-first launch order, default on; set only), and the testing hooks
 * "debug_outputs" (also write qfrc_bias, qfrc_smooth, qacc_smooth, qM, qfrc_constraint),
 * "dense_factor" (always take the dense factorisation schedule instead of the dof-tree one) and
 * "full_solver" (Newton on all dofs even when a leading block suffices).
 * Read only: "smem_bytes_per_env", "maxcon", "reduced_block_cap". Any other key is an error. */
int b2_set_option(b2_sim* sim, const char* key, double value);
int b2_get_option(b2_sim* sim, const char* key, double* value);

/* The hot path. */
int b2_step(b2_sim* sim, void* cuda_stream);              /* mjwarp.step    */
int b2_forward(b2_sim* sim, void* cuda_stream);           /* mjwarp.forward */
int b2_step_n(b2_sim* sim, int n, void* cuda_stream);     /* n sub-steps with ctrl held (decimation) */
/* forward() restricted to the worlds whose byte in `world_mask_dev` (device pointer, nworld bytes,
 * e.g. a torch.bool tensor) is non-zero: the partial-reset forward of manager_based_rl_env.py:128-132
 * without recomputing worlds that were not reset (SURVEY.md §8f-3). */
int b2_forward_masked(b2_sim* sim, const unsigned char* world_mask_dev, void* cuda_stream);

/* End-to-end call with HOST buffers (pinned or pageable): copies `ctrl` (nworld*nu floats, row
 * stride nu) to the device, runs `nsubstep` steps, copies qpos (nworld*nq) and qvel (nworld*nv)
 * back; asynchronous on `cuda_stream` when the host buffers are pinned. NULL outputs are skipped. */
int b2_step_host(b2_sim* sim, const float* ctrl_host, int nsubstep, float* qpos_host,
                 float* qvel_host, void* cuda_stream);

/* Fused MDP glue of the velocity-tracking task around the step (SURVEY.md §8f-1..3): what
 * ManagerBasedRlEnv.step (manager_based_rl_env.py:106-147) does before and after the decimation loop for
 * tasks/velocity/velocity_env_cfg.py, as two launches. All pointers are device pointers. */
#define B2_VELENV_NU(nu) (16 + 9 + 2 * (nu))
typedef struct B2VelEnvArgs {
  const float* action;            /* [n][nu] */
  const float* U;                 /* [n][B2_VELENV_NU(nu)] uniforms in [0,1): 0-1 reset xy, 2 yaw, 3-5 command, 6 heading
                                     target, 7 standing draw, 8 command timer, 9-10 push, 11 push timer, 12-15 spare,
                                     16.. observation noise (9 + 2 nu) */
  const float* default_qpos;      /* [nq] */
  const float* default_joint_pos; /* [nu] */
  const float* action_scale;      /* [nu] */
  const float* soft_lo;           /* [nu] */
  const float* soft_hi;           /* [nu] */
  const float* env_origins;       /* [n][3] */
  int32_t* episode_length;        /* [n] in/out */
  float* last_action;             /* [n][nu] in/out */
  float* command;                 /* [n][3] in/out */
  float* push_time_left;          /* [n] in/out */
  float* obs;                     /* [n][9 + 3 nu + 3] out */
  float* reward;                  /* [n] out */
  unsigned char* terminated;      /* [n] out */
  unsigned char* truncated;       /* [n] out */
  unsigned char* done;            /* [n] out: mask for b2_forward_masked */
  float* cmd_time_left;           /* [n] in/out: command resampling timer (velocity_env_cfg.py:69 3..8 s) */
  float* heading_target;          /* [n] in/out: heading command (velocity_command.py:71-75) */
  unsigned char* is_standing;     /* [n] in/out: standing envs get a zero command (rel_standing_envs = 0.1) */
  float* critic;                  /* [n][9 + 3 nu + 3] out: the same terms without noise (PrivilegedCfg) */
  float* log_row;                 /* [n][3] out: (reward, terminated, truncated) packed for the rank-0 log gather */
  float step_dt, fall_angle, push_vel, push_lo, push_hi;
  int32_t max_episode_length;
} B2VelEnvArgs;
int b2_velenv_pre(b2_sim* sim, const float* action, const float* default_joint_pos,
                  const float* action_scale, void* cuda_stream);
int b2_velenv_post(b2_sim* sim, const B2VelEnvArgs* args, void* cuda_stream);

/* ---- fused MDP glue of the motion-tracking task (BASELINE config C; reference tasks/tracking/tracking_env_cfg.py,
 * tasks/tracking/mdp/commands.py:283-388) ------------------------------------------------------------------------
 * post1 runs after the sub-steps (terminations, rewards, RSI resets, clip time step) and leaves the mask for
 * b2_forward_masked; post2 runs after that forward (anchor-relative targets, interval push, observations).
 * Per-step uniforms U[n][B2_TRACKENV_NU(nu)]: with S = 13 + nu, [0, S) reset block (0 clip frame, 1-6 pose noise,
 * 7-12 velocity noise, 13.. joint noise), [S, 2S) the same for envs that ran off the clip, [2S, 2S+7) push (6
 * velocity + timer), then observation noise: anchor pos 3, anchor ori 6, base lin 3, base ang 3, joint pos nu, joint vel nu. */
#define B2_TRACKENV_NU(nu) (48 + 4 * (nu))
typedef struct B2TrackEnvArgs {
  const float* action;            /* [n][nu] */
  const float* U;                 /* [n][B2_TRACKENV_NU(nu)] */
  const float* default_joint_pos; /* [nu] */
  const float* soft_lo;           /* [nu] */
  const float* soft_hi;           /* [nu] */
  const float* env_origins;       /* [n][3] */
  const float* m_joint_pos;       /* motion clip, T frames: [T][nu] */
  const float* m_joint_vel;       /* [T][nu] */
  const float* m_body_pos;        /* [T][nb][3] */
  const float* m_body_quat;       /* [T][nb][4] */
  const float* m_body_lin;        /* [T][nb][3] */
  const float* m_body_ang;        /* [T][nb][3] */
  const int32_t* body_idx;        /* [nb] engine body ids of the tracked bodies */
  const int32_t* ee_idx;          /* [nee] end effectors, as indices into the tracked bodies */
  int64_t* time_steps;            /* [n] in/out: clip frame */
  int32_t* episode_length;        /* [n] in/out */
  float* last_action;             /* [n][nu] in/out */
  float* push_time_left;          /* [n] in/out */
  float* body_pos_rel;            /* [n][nb][3] in/out: anchor-relative target positions */
  float* body_quat_rel;           /* [n][nb][4] in/out */
  float* reward;                  /* [n] out */
  unsigned char* terminated;      /* [n] out */
  unsigned char* truncated;       /* [n] out */
  unsigned char* mask;            /* [n] out: envs whose state was rewritten (reset or clip restart) */
  float* log_row;                 /* [n][3] out */
  float* obs;                     /* [n][5 nu + 15] out */
  float* critic;                  /* [n][5 nu + 15 + 9 nb] out */
  float pose_range[12], vel_range[12]; /* (lo, hi) x 6 */
  float step_dt, jp_lo, jp_hi, push_lo, push_hi;
  int32_t nb, nee, anchor, T, self_collision_adr, root_body, max_episode_length;
} B2TrackEnvArgs;
int b2_trackenv_post1(b2_sim* sim, const B2TrackEnvArgs* args, void* cuda_stream);
int b2_trackenv_post2(b2_sim* sim, const B2TrackEnvArgs* args, void* cuda_stream);

/* Diagnostics (synchronises `cuda_stream`). */
int b2_stats(b2_sim* sim, void* cuda_stream, B2Stats* out);
/* Number of kernels this library has launched for `sim` since creation. */
int64_t b2_launch_count(b2_sim* sim);
/* Algorithmic bytes of one step for the roofline (DESIGN.md): solver stage and whole step,
 * evaluated with the mean nefc of the last step. */
int b2_algorithmic_bytes(b2_sim* sim, void* cuda_stream, double* solver_bytes, double* step_bytes);

const char* b2_last_error(void);
const char* b2_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B2SIM_H_ */
