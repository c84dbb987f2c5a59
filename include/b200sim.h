/* b200sim C-ABI: the drop-in boundary of the CUDA path.
 *
 * The reference crosses into native code through the pybind11 module `mujoco`
 * (gymnasium_robotics/envs/robot_env.py:293-294 MjModel/MjData, :341 mj_step, fetch_env.py:303,401 mj_forward,
 * utils/mujoco_utils.py:115,125 mj_jacSite).  Those per-env, per-call entry points are replaced by the batched
 * entry points below: one call advances every env by one `step()` of the reference
 * (BaseRobotEnv.step, robot_env.py:114-152) entirely on the GPU.
 *
 * Conventions: opaque handle, int error codes (0 = ok), no exceptions, no torch types.  Every `float*`/`int*`
 * argument of step/refresh/raw_step is a DEVICE pointer owned by the caller ([N, dim] row-major, fp32); the
 * library owns the persistent per-env state.  Calls are asynchronous and ordered on `stream` (a cudaStream_t,
 * NULL = default stream).  `b200sim_last_error` returns a static or handle-owned string.
 */
#ifndef B200SIM_H
#define B200SIM_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200sim b200sim_t;

/* Task constants of the Fetch family (reference: envs/fetch/fetch_env.py:29-69 ctor args, resolved to ids). */
typedef struct b200sim_fetch_task {
  int has_object, block_gripper, n_substeps, reward_dense;
  int grip_site, obj_site, frame_site; /* site ids: "robot0:grip", "object0", frame of body robot0:gripper_link */
  int nrobot;                          /* joints whose name starts with "robot" (utils/mujoco_utils.py:23-31) */
  int robot_qadr[16], robot_dadr[16];
  int finger_qadr[2];                  /* qpos addresses zeroed by _step_callback when block_gripper */
  int nobs;
  float distance_threshold, dt;
  /* task family: 0 = Fetch (fields above), 1 = AntMaze (envs/maze/ant_maze_v5.py: ctrl = action, obs = qpos[2:]|qvel,
   * goal = xy; uses nobs, n_substeps (= frame_skip), reward_dense, nact, ngoal, success_radius) */
  int kind, nact, ngoal;
  float success_radius;
  int obs_qpos_start;   /* maze: first qpos entry inside `observation` (ant_maze_v5.py:312-320: 2; point_maze.py:404-410: 0) */
  float vel_clip;       /* maze: |qvel| clip before stepping (envs/maze/point.py:73-77: 5.0; 0 = none) */
  /* kind 2 = Shadow-hand manipulation (envs/shadow_dexterous_hand/hand_env.py:42-61 absolute control, manipulate.py:88-138,
   * 298-314): nact = 20, ngoal = 7, obs = robot qpos | robot qvel | object qvel | object qpos; obj_qadr / obj_dadr = qpos /
   * dof address of "object:joint" (must be the last joint); goal_flags bit 0: position counts, bit 1: rotation counts */
  int obj_qadr, obj_dadr, goal_flags;
  float rotation_threshold;
  /* touch observation appended after the 61 base entries (manipulate_touch_sensors.py:107-138): 0 = none,
   * 1 = sensordata, 2 = boolean, 3 = log(x + 1); one value per touch sensor of the model.
   * kind 1 (maze agents): 1 = append the clipped per-body contact forces of Gymnasium's Ant-v5 (`cfrc_ext[1:]`, 6 per body,
   * [torque; force] about the tree root's subtree com, clipped to (-1, 1)): the (105,) observation of AntMaze_*-v5
   * (envs/maze/ant_maze_v5.py:99, 132-134); 0 = the (27,) observation of AntMaze_*-v4 / PointMaze */
  int touch_mode;
  /* kind 3 = HandReach (envs/shadow_dexterous_hand/reach.py): same control as kind 2, obs = robot qpos | robot qvel |
   * 5 fingertip site positions = achieved goal (ngoal = 15), Fetch-style distance reward with distance_threshold */
  int tip_site[5];
  /* kind 4 = AdroitHandHammer (envs/adroit_hand/adroit_hammer.py:291-357): absolute control as kind 2, frame_skip sub-steps,
   * obs = qpos[:-6] | clip(qvel[-6:]) | palm | hammer pos | hammer euler | nail | clip(touch "S_nail") (46), dense / sparse
   * reward, success = nail within 1 cm of its goal.  Sites: grip_site = "S_grasp", obj_site = body frame of "Object",
   * frame_site = "S_target", tip_site[0] = "tool", tip_site[1] = "nail_goal".
   * penv_body: runtime body whose body_pos is per-env state (nail_board, adroit_hammer.py:372-378), -1 = none; its pose (position
   * 3 + quaternion 4 floats) lives in the state record at B200SIM_ST_PENV. */
  /* kind 5 = AdroitHandRelocate (envs/adroit_hand/adroit_relocate.py:288-373): obs = qpos[:-6] | palm - ball | palm - target |
   * ball - target (39); grip_site = "S_grasp", obj_site = body frame of "Object", penv_body = "Object" (body_pos x, y redrawn per
   * episode), the per-env target site position is the 3-float goal of the state record. */
  /* kind 6 = AdroitHandPen (envs/adroit_hand/adroit_pen.py:288-378): obs 45; obj_site = body frame of "Object", frame_site =
   * "eps_ball", tip_site[0..3] = object_top, object_bottom, target_top, target_bottom; distance_threshold = pen length,
   * rotation_threshold = target length (:392-399); penv_body = "target" (body_quat redrawn per episode, :379-384). */
  /* kind 7 = AdroitHandDoor (envs/adroit_hand/adroit_door.py:279-371): obs 39; grip_site = "S_grasp", frame_site = "S_handle",
   * obj_qadr = qpos address of "door_hinge", penv_body = "frame" (body_pos redrawn per episode). */
  /* kind 8 = FrankaKitchen (envs/franka_kitchen/franka_env.py:92-128, kitchen_env.py:371-397): the action is the clipped
   * position target of the nact = nu actuators (the caller derives it from the last noisy observation, franka_env.py:139-170),
   * n_substeps = 40; obs = robot qpos | robot qvel | object qpos | object qvel (nq + nv, noise-free: the caller adds the
   * observation noise), achieved = qpos (ngoal = nq; the per-task slices of kitchen_env.py:27-45 are taken by the caller),
   * reward 0.  Chosen together with the bring-up kernel build for models with joint equalities / condim 6. */
  int penv_body;
} b200sim_fetch_task_t;

/* indices into the layout array returned by b200sim_layout (offsets in floats inside one env's state record) */
enum { B200SIM_ST_QPOS = 0, B200SIM_ST_QVEL, B200SIM_ST_WARM, B200SIM_ST_CTRL, B200SIM_ST_MOCAP, B200SIM_ST_POSE,
       B200SIM_ST_GOAL, B200SIM_ST_STRIDE, B200SIM_ST_PENV, B200SIM_ST_COUNT };

/* model_blob: include/b200sim_model.h format.  eq_data: NULL, or exactly [neq*11] doubles overriding the model's equality data
 * (the reference rewrites it after load: utils/mujoco_utils.py:74-80); the library cannot see its length.  ref: fixed world point the spatial algebra is
 * expressed about.  Replaces MjModel.from_xml_path + MjData (robot_env.py:293-294). */
int b200sim_create(const void* model_blob, size_t nbytes, const double* eq_data, const float* ref,
                   const b200sim_fetch_task_t* task, int num_envs, int device, b200sim_t** out);
void b200sim_destroy(b200sim_t* h);
const char* b200sim_last_error(const b200sim_t* h);

int b200sim_num_envs(const b200sim_t* h);
int b200sim_layout(const b200sim_t* h, int* out /* [B200SIM_ST_COUNT] */);
/* device pointer to the [num_envs, stride] fp32 state records (qpos|qvel|qacc_warmstart|ctrl|mocap|pose|goal) --
 * the hook for reset, parity injection and checkpointing (reference: data.qpos/qvel views, robot_env.py:301-315). */
float* b200sim_state(b200sim_t* h);

/* One env.step() for every env: clip + _set_action + n_substeps x mj_step + _step_callback + _get_obs + reward, plus the episode
 * bookkeeping of the step (BaseRobotEnv.compute_terminated / compute_truncated, robot_env.py:106-112, 143-146, and gymnasium's
 * TimeLimit wrapper): terminated / truncated (optional, [N] bytes each) -- see b200sim_set_time_limit.
 * info (optional, [N] int32): low 16 bits = Newton iterations spent, bit 16.. = capacity-overflow flags. */
int b200sim_step(b200sim_t* h, const float* actions, float* obs, float* achieved, float* desired, float* reward, float* success,
                 unsigned char* terminated, unsigned char* truncated, int* info, void* stream);
/* TimeLimit inside the step kernel: the library owns one step counter per env (device, [N] int32, b200sim_elapsed) that a
 * b200sim_step launch increments and the b200sim_reset* draws zero; truncated = counter >= max_episode_steps (<= 0: never).
 * terminate_on_success != 0: terminated = success (MazeEnv.compute_terminated with continuing_task = False, maze_v4.py:390-398);
 * 0: terminated = False (Fetch / Hand / Adroit).  Callers that write state records themselves also zero the counters they reset. */
int b200sim_set_time_limit(b200sim_t* h, int max_episode_steps, int terminate_on_success);
int* b200sim_elapsed(b200sim_t* h);
/* device counter (one unsigned 64-bit word): env-steps so far in which a capacity limit dropped candidates / contacts / rows */
unsigned long long* b200sim_overflow_counter(b200sim_t* h);
/* Packed output rows: after b200sim_set_packed(h, 1) every entry point that takes (obs, achieved, desired, reward, success)
 * expects `obs` to point at ONE [N, W] fp32 buffer, W = b200sim_packed_width(h), and ignores the other four pointers.
 * Row layout: obs[nobs] | achieved[ngoal] | desired[ngoal] | reward | success | terminated | truncated | pad (W is a multiple
 * of 4 floats; the two flags are 0.0 / 1.0).  One device->host copy or one all-gather then moves everything a step produced. */
int b200sim_packed_width(const b200sim_t* h);
int b200sim_set_packed(b200sim_t* h, int enable);
/* mj_forward-style refresh of derived quantities + observation for envs with mask[i] != 0 (mask NULL = all);
 * used after reset writes new state records (reference: fetch_env.py:375-402 _reset_sim -> mj_forward, _get_obs). */
int b200sim_refresh(b200sim_t* h, const unsigned char* mask, float* obs, float* achieved, float* desired, float* reward,
                    float* success, void* stream);
/* nstep raw mj_step calls with the ctrl / mocap currently in the state records (reference: fetch_env.py:419-420). */
int b200sim_raw_step(b200sim_t* h, int nstep, float* obs, float* achieved, float* desired, float* reward, float* success,
                     void* stream);
/* the same for envs with mask[i] != 0 only (mask NULL = all): the settle phase of a partial reset
 * (reference: envs/shadow_dexterous_hand/manipulate.py:213-222, 10 x mj_step(nstep=n_substeps) inside _reset_sim). */
int b200sim_raw_step_masked(b200sim_t* h, const unsigned char* mask, int nstep, float* obs, float* achieved, float* desired,
                            float* reward, float* success, void* stream);
/* Draw parameters of a Fetch reset (reference: envs/fetch/fetch_env.py:375-402 _reset_sim, :153-166 _sample_goal; the values the
 * reference keeps on the env object: obj_range, target_range, target_offset, target_in_the_air, height_offset,
 * initial_gripper_xpos); obj_qadr = qpos address of "object0:joint". */
typedef struct b200sim_fetch_reset {
  int has_object, target_in_the_air, obj_qadr;
  float obj_range, target_range, target_offset[3], height_offset, gripper_xpos[3];
} b200sim_fetch_reset_t;
/* In-kernel reset of the envs with mask[i] != 0 (mask NULL = all), Fetch task family: the env's state record becomes
 * `rest_record` (device, [stride] floats: mj_resetData + initial qpos / qvel / mocap, fetch_env.py:376-381) with the object start
 * and the goal drawn on the device -- Philox4x32-10 keyed by `seed`, counter (env index + env_offset, episode[i]) -- followed by
 * mj_forward + _get_obs exactly as b200sim_refresh.  `episode` (device, [N] int32, may be NULL = episode 0) holds per-env
 * episode counters and is incremented for the reset envs, so that consecutive resets of an env never repeat a draw;
 * `env_offset` is the global index of this handle's first env (sharded runs draw what one big batch would draw).
 * Replaces the per-env np_random draws of BaseRobotEnv.reset (robot_env.py:154-186) in the throughput RNG mode. */
int b200sim_reset(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_fetch_reset_t* params,
                  unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired, float* reward,
                  float* success, void* stream);
/* The same for reset_model functions that are a fixed list of uniform draws (any task family; reference:
 * adroit_hammer.py:372-378, adroit_relocate.py:354-373, adroit_door.py:359-371): record <- rest_record, then
 * record[slot[k]] = lo[k] + (hi[k] - lo[k]) * u_k for k < n (u_k: word k % 4 of Philox block k / 4), then the refresh.
 * A draw with slot -1 - j (j = 0..2) is Euler angle j of an orientation instead: when quat_slot >= 0 the four floats at quat_slot
 * become euler2quat(angles) (utils/rotations.py:87-113; adroit_pen.py:379-384 draws the target pen's orientation this way). */
#define B200SIM_RESET_SLOTS_MAX 16
typedef struct b200sim_uniform_reset {
  int n, slot[B200SIM_RESET_SLOTS_MAX];   /* offsets in floats inside the state record (b200sim_layout) */
  float lo[B200SIM_RESET_SLOTS_MAX], hi[B200SIM_RESET_SLOTS_MAX];
  int quat_slot;                          /* -1 = none */
} b200sim_uniform_reset_t;
int b200sim_reset_uniform(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_uniform_reset_t* params,
                          unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired,
                          float* reward, float* success, void* stream);
/* Maze family (AntMaze / PointMaze; reference: envs/maze/maze_v4.py:256-297, 299-373): goal cell + noise, reset cell farther than
 * half a cell from the goal + noise.  goal_xy / reset_xy: DEVICE tables [n_goal, 2] / [n_reset, 2] of cell centres
 * (MazeEnv.maze.unique_goal_locations / unique_reset_locations, or all free cells when the map marks none, maze_v4.py:212-228). */
typedef struct b200sim_maze_reset {
  int n_goal, n_reset;
  float scaling, noise;   /* maze_size_scaling; position_noise_range (0.25) */
} b200sim_maze_reset_t;
int b200sim_reset_maze(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_maze_reset_t* params,
                       const float* goal_xy, const float* reset_xy, unsigned long long seed, int env_offset, int* episode, float* obs,
                       float* achieved, float* desired, float* reward, float* success, void* stream);
/* Shadow-Hand manipulation (reference: envs/shadow_dexterous_hand/manipulate.py:154-224 _reset_sim, :226-279 _sample_goal).  The
 * reference's reset is a retry loop, so the draws are two calls: `b200sim_reset_hand_pose` writes rest_record + the drawn object
 * start pose into the masked envs' records (their goal survives) for attempt number `attempt` -- the caller then settles with
 * b200sim_raw_step_masked and repeats for the envs whose object left the palm; `b200sim_reset_hand_goal` draws the goal from the
 * settled object pose, increments episode[i] and refreshes.  rot modes: 0 none, 1 "z", 2 "parallel", 3 "xyz"; parallel_quats is the
 * DEVICE table [24, 4] of rotations.get_parallel_rotations() (utils/rotations.py:349-386). */
typedef struct b200sim_hand_reset {
  int obj_qadr, rot_mode, randomize_rotation, randomize_position, goal_rot_mode, goal_random_position;
  float pos_lo[3], pos_hi[3];   /* manipulate.py: target_position_range */
} b200sim_hand_reset_t;
int b200sim_reset_hand_pose(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_hand_reset_t* params,
                            const float* parallel_quats, unsigned long long seed, int env_offset, const int* episode, int attempt,
                            void* stream);
int b200sim_reset_hand_goal(b200sim_t* h, const unsigned char* mask, const b200sim_hand_reset_t* params, const float* parallel_quats,
                            unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired,
                            float* reward, float* success, void* stream);
/* HandReach (reference: envs/shadow_dexterous_hand/reach.py:95-130): record <- rest_record with the 15-float goal drawn on the
 * device (meeting point of the thumb and a random other finger tip), then the refresh.  meeting = palm_xpos + (0, -0.09, 0.05). */
typedef struct b200sim_reach_reset { float meeting[3], initial_goal[15]; } b200sim_reach_reset_t;
int b200sim_reset_reach(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_reach_reset_t* params,
                        unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired, float* reward,
                        float* success, void* stream);
/* Failure detection ([ext] mj_checkPos / mj_checkVel / mj_checkAcc inside mj_step: NaN or |x| > 1e10 => warning + mj_resetData):
 * bad[i] (device, [N] bytes) = 1 when env i's state record holds a non-finite or huge value, else 0.  With rest_record != NULL a bad
 * env's record is replaced by it, except the float ranges listed in `keep` (goal, per-episode poses) whose finite values survive.
 * The caller follows with b200sim_refresh(mask = bad) to recompute the observation of the recovered envs. */
typedef struct b200sim_keep { int n, start[4], len[4]; } b200sim_keep_t;
int b200sim_check_state(b200sim_t* h, unsigned char* bad, const float* rest_record, const b200sim_keep_t* keep, void* stream);
/* GoalEnv.compute_reward on M (achieved, desired) pairs, device pointers (reference: fetch_env.py:74-80). */
int b200sim_compute_reward(const b200sim_t* h, const float* achieved, const float* desired, int M, float* out, void* stream);
/* number of kernel launches issued through this handle so far */
long b200sim_launch_count(const b200sim_t* h);
/* shared-memory bytes per block and warps (envs) per block chosen at create time */
int b200sim_launch_config(const b200sim_t* h, int* smem_bytes, int* envs_per_block, int* blocks);
/* which step-kernel instantiation this handle launches: envs per block, the padded dof count NVP of the template, and the build
 * (translation unit) it lives in.  Read-only; any pointer may be NULL. */
enum { B200SIM_BUILD_ARM = 0,            /* b200sim.cu: Fetch, mazes, Shadow Hand, Adroit up to 30 dofs */
       B200SIM_BUILD_WIDE = 1,           /* b200sim_wide.cu: 33..36 dofs */
       B200SIM_BUILD_KITCHEN_FLAT = 2,   /* b200sim_kitchen.cu (B200SIM_KITCHEN_GROUPS=0) */
       B200SIM_BUILD_KITCHEN_GROUPS = 3, /* b200sim_kitchen_groups.cu */
       B200SIM_BUILD_KITCHEN_HULL = 4 }; /* b200sim_kitchen_hull.cu */
int b200sim_kernel_variant(const b200sim_t* h, int* envs_per_block, int* nvp, int* build);

#ifdef __cplusplus
}
#endif
#endif
