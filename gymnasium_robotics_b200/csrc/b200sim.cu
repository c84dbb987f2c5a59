// b200sim: CUDA kernels (sm_100a) + the C-ABI of include/b200sim.h.
//
// One warp integrates one env for a whole env-step (all sub-steps on chip); WPB warps share one copy of the model
// constants that a single thread stages into shared memory with a TMA bulk copy (cp.async.bulk + mbarrier).
// Per-env state lives in HBM as one contiguous fp32 record per env (read once, written once per step).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string>
#include <vector>

#include "../../include/b200sim.h"
#include "step_kernel.cuh"
#include "reset_sample.cuh"

// warps (= envs) per block: 28 fills an SM in one wave at 4096 envs per GPU; smaller batches use smaller blocks so
// that every SM still gets work (e.g. the 1024-env shards of BASELINE config 4)
#define B200_WPB_MAX 28

#ifdef B200_STAGE_TIMING
extern "C" int b200sim_debug_stage_cycles(unsigned long long* out, int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, g_stage_cycles, sizeof(unsigned long long) * TM_COUNT);
  if (reset) { unsigned long long z[TM_COUNT] = {0}; cudaMemcpyToSymbol(g_stage_cycles, z, sizeof(z)); }
  return TM_COUNT;
}
#endif

__global__ void reward_kernel(const float* __restrict__ ag, const float* __restrict__ dg, int M, int ngoal, int kind, float thr,
                              float radius, int dense, FetchTask task, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  if (kind == TASK_HAND) {   // manipulate.py:120-128
    float dp, dr;
    hand_goal_distance(task, ag + 7 * i, dg + 7 * i, &dp, &dr);
    out[i] = hand_reward(task, dp, dr, nullptr);
    return;
  }
  float d2 = 0;
  for (int k = 0; k < ngoal; k++) { float e = ag[ngoal * i + k] - dg[ngoal * i + k]; d2 = fmaf(e, e, d2); }   // (explicit: see antmaze_observe)
  float d = sqrtf(d2);
  if (kind == TASK_FETCH || kind == TASK_HAND_REACH) out[i] = dense ? -d : -(d > thr ? 1.f : 0.f);   // fetch_env.py:74-80, reach.py:88-93
  else out[i] = dense ? expf(-d) : (d <= radius ? 1.f : 0.f);               // maze_v4.py:381-388
}

// in-kernel reset draw (reset_sample.cuh): one thread per env writes its state record; the refresh launch that follows does
// mj_forward + _get_obs.  32 consecutive threads write 32 consecutive records word by word (stride ~ 60 words: each record is
// a few 128-byte lines, touched once per episode).
__global__ void fetch_reset_kernel(b200sim_fetch_reset_t p, unsigned long long seed, int env_offset, int N, const unsigned char* __restrict__ mask,
                                   const float* __restrict__ rest, int stride, int st_qpos, int st_goal, float* __restrict__ state,
                                   int* __restrict__ episode, int* __restrict__ elapsed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (mask && !mask[i])) return;
  int ep = episode ? episode[i] : 0;
  rs_fetch_reset_record(p, seed, (uint32_t)(i + env_offset), (uint32_t)ep, rest, stride, st_qpos, st_goal, state + (size_t)i * stride);
  if (episode) episode[i] = ep + 1;
  if (elapsed) elapsed[i] = 0;   // a reset env starts a new episode of the TimeLimit
}

__global__ void uniform_reset_kernel(b200sim_uniform_reset_t p, unsigned long long seed, int env_offset, int N, const unsigned char* __restrict__ mask,
                                     const float* __restrict__ rest, int stride, float* __restrict__ state, int* __restrict__ episode, int* __restrict__ elapsed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (mask && !mask[i])) return;
  int ep = episode ? episode[i] : 0;
  rs_uniform_reset_record(p, seed, (uint32_t)(i + env_offset), (uint32_t)ep, rest, stride, state + (size_t)i * stride);
  if (episode) episode[i] = ep + 1;
  if (elapsed) elapsed[i] = 0;   // a reset env starts a new episode of the TimeLimit
}

__global__ void maze_reset_kernel(b200sim_maze_reset_t p, const float* __restrict__ goal_xy, const float* __restrict__ reset_xy, unsigned long long seed,
                                  int env_offset, int N, const unsigned char* __restrict__ mask, const float* __restrict__ rest, int stride,
                                  int st_qpos, int st_goal, float* __restrict__ state, int* __restrict__ episode, int* __restrict__ elapsed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (mask && !mask[i])) return;
  int ep = episode ? episode[i] : 0;
  rs_maze_reset_record(p, goal_xy, reset_xy, seed, (uint32_t)(i + env_offset), (uint32_t)ep, rest, stride, st_qpos, st_goal, state + (size_t)i * stride);
  if (episode) episode[i] = ep + 1;
  if (elapsed) elapsed[i] = 0;   // a reset env starts a new episode of the TimeLimit
}

__global__ void check_state_kernel(int N, int stride, float* __restrict__ state, const float* __restrict__ rest, b200sim_keep_t keep,
                                   unsigned char* __restrict__ bad) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  bad[i] = (unsigned char)rs_check_record(state + (size_t)i * stride, stride, rest, keep);
}

__global__ void hand_pose_kernel(b200sim_hand_reset_t p, const float* __restrict__ parallel, unsigned long long seed, int env_offset, int N,
                                 const unsigned char* __restrict__ mask, const float* __restrict__ rest, int stride, int st_qpos, int st_goal,
                                 int ngoal, float* __restrict__ state, const int* __restrict__ episode, int attempt) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (mask && !mask[i])) return;
  rs_hand_pose_record(p, parallel, seed, (uint32_t)(i + env_offset), (uint32_t)(episode ? episode[i] : 0), (uint32_t)attempt, rest, stride, st_qpos,
                      st_goal, ngoal, state + (size_t)i * stride);
}
__global__ void hand_goal_kernel(b200sim_hand_reset_t p, const float* __restrict__ parallel, unsigned long long seed, int env_offset, int N,
                                 const unsigned char* __restrict__ mask, int stride, int st_qpos, int st_goal, float* __restrict__ state,
                                 int* __restrict__ episode, int* __restrict__ elapsed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (mask && !mask[i])) return;
  int ep = episode ? episode[i] : 0;
  rs_hand_goal(p, parallel, seed, (uint32_t)(i + env_offset), (uint32_t)ep, st_qpos, st_goal, state + (size_t)i * stride);
  if (episode) episode[i] = ep + 1;
  if (elapsed) elapsed[i] = 0;   // a reset env starts a new episode of the TimeLimit
}

__global__ void reach_reset_kernel(b200sim_reach_reset_t p, unsigned long long seed, int env_offset, int N, const unsigned char* __restrict__ mask,
                                   const float* __restrict__ rest, int stride, int st_goal, float* __restrict__ state, int* __restrict__ episode, int* __restrict__ elapsed) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (mask && !mask[i])) return;
  int ep = episode ? episode[i] : 0;
  rs_reach_reset_record(p, seed, (uint32_t)(i + env_offset), (uint32_t)ep, rest, stride, st_goal, state + (size_t)i * stride);
  if (episode) episode[i] = ep + 1;
  if (elapsed) elapsed[i] = 0;   // a reset env starts a new episode of the TimeLimit
}

// ---------------------------------------------------------------------------------------------------------------
#define B200_FOR_ALL_VARIANTS(X) X(7, 14) X(7, 15) X(7, 21) X(14, 14) X(14, 15) X(14, 21) X(28, 14) X(28, 15) X(28, 21) \
  X(7, 22) X(14, 22) X(28, 22) X(7, 30) X(14, 30)

// wide build (models with 33..40 dofs), compiled from b200sim_wide.cu with 64-bit dof masks
extern "C" int b200sim_wide_setattr(int wpb, int smem_bytes);
extern "C" int b200sim_wide_launch(int wpb, int blocks, size_t smem_bytes, void* stream, const uint32_t* model_dev, const FetchTask* task,
                                   int mode, int nraw, int N, const StepIO* io);
#define B200_WIDE_NVP 36
// build for models with joint equalities / condim 6 (Franka Kitchen), compiled from b200sim_kitchen.cu (flat broad-phase scan) and
// b200sim_kitchen_groups.cu (two-level broad phase; the default, B200SIM_KITCHEN_GROUPS=0 selects the flat scan)
extern "C" int b200sim_kitchen_build(const b200_model_view* view, const double* eq_data, const float* ref, int penv_body,
                                     std::vector<uint32_t>* buf, std::string* err);
extern "C" int b200sim_kitchen_setattr(int wpb, int smem_bytes);
extern "C" int b200sim_kitchen_groups_build(const b200_model_view* view, const double* eq_data, const float* ref, int penv_body,
                                            std::vector<uint32_t>* buf, std::string* err);
extern "C" int b200sim_kitchen_groups_setattr(int wpb, int smem_bytes);
extern "C" int b200sim_kitchen_groups_launch(int wpb, int blocks, size_t smem_bytes, void* stream, const uint32_t* model_dev, const FetchTask* task,
                                             int mode, int nraw, int N, const StepIO* io);
// b200sim_kitchen_hull.cu: the groups build + support-map narrow phase for MESH geoms (models compiled with mesh_hull)
extern "C" int b200sim_kitchen_hull_build(const b200_model_view* view, const double* eq_data, const float* ref, int penv_body,
                                          std::vector<uint32_t>* buf, std::string* err);
extern "C" int b200sim_kitchen_hull_setattr(int wpb, int smem_bytes);
extern "C" int b200sim_kitchen_hull_launch(int wpb, int blocks, size_t smem_bytes, void* stream, const uint32_t* model_dev, const FetchTask* task,
                                             int mode, int nraw, int N, const StepIO* io);
extern "C" int b200sim_kitchen_launch(int wpb, int blocks, size_t smem_bytes, void* stream, const uint32_t* model_dev, const FetchTask* task,
                                      int mode, int nraw, int N, const StepIO* io);
#define B200_KITCHEN_NVP 31   // the kitchen translation unit instantiates NVP = 31 (identity-padded; distinct kernel symbols)

struct b200sim {
  int N = 0, device = 0;
  bool kitchen = false, kitchen_groups = false, hull = false;
  std::vector<uint8_t> blob;
  b200_model_view view;
  std::vector<uint32_t> model_host;
  uint32_t* model_dev = nullptr;
  FetchTask task;
  float* state = nullptr;
  int* elapsed = nullptr;                        // per-env step counters of the TimeLimit (device, [N])
  unsigned long long* overflow_count = nullptr;  // env-steps that hit a capacity limit (device counter)
  int max_steps = 0, term_on_success = 0;        // b200sim_set_time_limit
  int packed = 0, packed_w = 0;                  // b200sim_set_packed
  size_t smem_bytes = 0;
  int blocks = 0;
  long launches = 0;
  int nvp = 32, wpb = B200_WPB_MAX;
  std::string err;
};

static std::string g_err;

static int fail(b200sim* h, const std::string& msg, int code) {
  if (h) h->err = msg; else g_err = msg;
  return code;
}

#define CUDA_OK(call)                                                                                         \
  do {                                                                                                        \
    cudaError_t e_ = (call);                                                                                  \
    if (e_ != cudaSuccess) return fail(h, std::string(#call) + ": " + cudaGetErrorString(e_), -100 - (int)e_); \
  } while (0)

// every entry point runs on the handle's device and leaves the caller's current device as it found it
struct DevGuard {
  int prev = -1; bool ok = true;
  explicit DevGuard(int dev) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess; }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ON_DEVICE(h) DevGuard guard_((h)->device); if (!guard_.ok) return fail(h, "cudaSetDevice failed", -7)

static void free_handle(b200sim* h) {
  if (!h) return;
  if (h->model_dev) cudaFree(h->model_dev);
  if (h->state) cudaFree(h->state);
  if (h->elapsed) cudaFree(h->elapsed);
  if (h->overflow_count) cudaFree(h->overflow_count);
  delete h;
}

extern "C" {

int b200sim_create(const void* model_blob, size_t nbytes, const double* eq_data, const float* ref,
                   const b200sim_fetch_task_t* task, int num_envs, int device, b200sim_t** out) {
  b200sim* h = nullptr;
  if (!model_blob || !task || !out || num_envs <= 0) return fail(nullptr, "b200sim_create: bad arguments", -1);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return fail(nullptr, "b200sim_create: no CUDA device (the CUDA path has no CPU fallback)", -2);
  h = new b200sim;
  h->N = num_envs; h->device = device;
  h->blob.assign((const uint8_t*)model_blob, (const uint8_t*)model_blob + nbytes);
  if (b200_model_parse(h->blob.data(), nbytes, &h->view) != 0) { delete h; return fail(nullptr, "b200sim_create: not a model blob", -3); }
  float r[3] = {0, 0, 0};
  if (ref) { r[0] = ref[0]; r[1] = ref[1]; r[2] = ref[2]; }
  std::string err;
  {
    // models with joint equalities or condim-6 pairs go to the bring-up translation unit (its contact records are larger)
    const b200_model_view& v = h->view;
    for (int e = 0; e < v.neq; e++) if (v.eq_type[e] == B200_EQ_JOINT) h->kitchen = true;
    for (int p = 0; p < v.npair; p++) if (v.pair_condim[p] == 6) h->kitchen = true;
  }
  const int penv = TASK_IS_ADROIT(task->kind) ? task->penv_body : -1;
  if (h->kitchen) { const char* g = getenv("B200SIM_KITCHEN_GROUPS"); h->kitchen_groups = !(g && g[0] && atoi(g) == 0); }  // default: two-level broad phase
  // MESH geoms (a model compiled with mesh_hull: hull vertex tables instead of box proxies) exist in the hull build only; that build
  // is the kitchen groups build plus the support-map narrow phase, so it serves any model the kitchen build serves
  for (int g = 0; g < h->view.ngeom; g++) if (h->view.geom_type[g] == B200_GEOM_MESH) h->hull = true;
  if (h->hull) { h->kitchen = true; h->kitchen_groups = true; }
  if ((h->kitchen ? (h->hull ? b200sim_kitchen_hull_build(&h->view, eq_data, r, penv, &h->model_host, &err)
                             : (h->kitchen_groups ? b200sim_kitchen_groups_build(&h->view, eq_data, r, penv, &h->model_host, &err)
                                                  : b200sim_kitchen_build(&h->view, eq_data, r, penv, &h->model_host, &err)))
                  : dm_build(h->view, eq_data, r, h->model_host, err, penv)) != 0) {
    delete h; return fail(nullptr, "b200sim_create: " + err, -4);
  }
  const DMHead* dh = (const DMHead*)h->model_host.data();
  FetchTask& t = h->task;
  memset(&t, 0, sizeof(t));
  t.has_object = task->has_object; t.block_gripper = task->block_gripper; t.n_substeps = task->n_substeps;
  t.reward_dense = task->reward_dense; t.grip_site = task->grip_site; t.obj_site = task->obj_site; t.frame_site = task->frame_site;
  t.nrobot = task->nrobot;
  if (task->kind == TASK_FETCH && (t.nrobot < 2 || t.nrobot > FETCH_MAX_ROBOT_JNT)) { delete h; return fail(nullptr, "b200sim_create: bad nrobot", -5); }
  for (int i = 0; i < 16; i++) { t.robot_qadr[i] = task->robot_qadr[i]; t.robot_dadr[i] = task->robot_dadr[i]; }
  t.finger_qadr[0] = task->finger_qadr[0]; t.finger_qadr[1] = task->finger_qadr[1];
  t.nobs = task->nobs; t.distance_threshold = task->distance_threshold; t.dt = task->dt;
  t.kind = task->kind; t.nact = task->nact; t.ngoal = task->ngoal; t.success_radius = task->success_radius;
  t.obs_qpos_start = task->obs_qpos_start; t.vel_clip = task->vel_clip;
  t.obj_qadr = task->obj_qadr; t.obj_dadr = task->obj_dadr; t.goal_flags = task->goal_flags; t.rotation_threshold = task->rotation_threshold;
  t.touch_mode = task->touch_mode;
  for (int k = 0; k < 5; k++) t.tip_site[k] = task->tip_site[k];
  t.penv_body = TASK_IS_ADROIT(task->kind) ? task->penv_body : -1;
  if (t.kind == TASK_FETCH) { t.nact = 4; t.ngoal = 3; }
  if (t.kind == TASK_ADROIT_HAMMER) {
    bool ok = t.nact == dh->nu && t.ngoal == 3 && t.nobs == dh->nq - 6 + 6 + 13 && dh->nsensor <= 1 && t.penv_body > 0 && t.penv_body < dh->nb;
    const int sites[5] = {t.grip_site, t.obj_site, t.frame_site, t.tip_site[0], t.tip_site[1]};
    for (int k = 0; k < 5; k++) ok = ok && sites[k] >= 0 && sites[k] < dh->nsite;
    if (!ok) { delete h; return fail(nullptr, "b200sim_create: inconsistent AdroitHandHammer task", -6); }
  }
  if (t.kind == TASK_ADROIT_DOOR) {
    bool ok = t.nact == dh->nu && t.ngoal == 3 && t.nobs == dh->nq - 3 + 12 && t.penv_body > 0 && t.penv_body < dh->nb &&
              t.obj_qadr >= 0 && t.obj_qadr < dh->nq && t.grip_site >= 0 && t.grip_site < dh->nsite && t.frame_site >= 0 && t.frame_site < dh->nsite;
    if (!ok) { delete h; return fail(nullptr, "b200sim_create: inconsistent AdroitHandDoor task", -6); }
  }
  if (t.kind == TASK_ADROIT_PEN) {
    bool ok = t.nact == dh->nu && t.ngoal == 3 && t.nobs == dh->nq - 6 + 21 && t.penv_body > 0 && t.penv_body < dh->nb &&
              t.distance_threshold > 0 && t.rotation_threshold > 0;
    const int sites[6] = {t.obj_site, t.frame_site, t.tip_site[0], t.tip_site[1], t.tip_site[2], t.tip_site[3]};
    for (int k = 0; k < 6; k++) ok = ok && sites[k] >= 0 && sites[k] < dh->nsite;
    if (!ok) { delete h; return fail(nullptr, "b200sim_create: inconsistent AdroitHandPen task", -6); }
  }
  if (t.kind == TASK_ADROIT_RELOCATE) {
    bool ok = t.nact == dh->nu && t.ngoal == 3 && t.nobs == dh->nq - 6 + 9 && t.penv_body > 0 && t.penv_body < dh->nb &&
              t.grip_site >= 0 && t.grip_site < dh->nsite && t.obj_site >= 0 && t.obj_site < dh->nsite;
    if (!ok) { delete h; return fail(nullptr, "b200sim_create: inconsistent AdroitHandRelocate task", -6); }
  }
  if (t.kind == TASK_KITCHEN) {
    if (!(h->kitchen && t.nact == dh->nu && t.ngoal == dh->nq && t.nobs == dh->nq + dh->nv)) { delete h; return fail(nullptr, "b200sim_create: inconsistent FrankaKitchen task", -6); }
  } else if (h->kitchen) { delete h; return fail(nullptr, "b200sim_create: this model needs the kitchen task kind (8)", -6); }
  if (t.kind != TASK_FETCH && t.kind != TASK_ANTMAZE && t.kind != TASK_HAND && t.kind != TASK_HAND_REACH && !TASK_IS_ADROIT(t.kind) && t.kind != TASK_KITCHEN) { delete h; return fail(nullptr, "b200sim_create: unknown task kind", -6); }
  if (t.kind == TASK_HAND && (t.nact != dh->nu || t.ngoal != 7 || t.obj_qadr != dh->nq - 7 || t.obj_dadr != dh->nv - 6 ||
                              t.touch_mode < 0 || t.touch_mode > 3 || (t.touch_mode && dh->nsensor == 0) ||
                              t.nobs != t.obj_qadr + dh->nv + 7 + (t.touch_mode ? dh->nsensor : 0))) { delete h; return fail(nullptr, "b200sim_create: inconsistent Hand task", -6); }
  if (t.kind == TASK_FETCH && dh->nmocap != 1) { delete h; return fail(nullptr, "b200sim_create: Fetch task needs exactly one mocap body", -6); }
  if (t.kind == TASK_ANTMAZE && (t.nact != dh->nu || t.ngoal != 2 || t.touch_mode < 0 || t.touch_mode > 1 ||
                                 t.nobs != dh->nq - t.obs_qpos_start + dh->nv + (t.touch_mode == 1 ? 6 * (dh->nmjb - 1) : 0))) { delete h; return fail(nullptr, "b200sim_create: inconsistent AntMaze task", -6); }
  if (t.kind == TASK_HAND_REACH) {
    bool ok = t.nact == dh->nu && t.ngoal == 15 && t.nobs == dh->nq + dh->nv + 15;
    for (int k = 0; k < 5; k++) ok = ok && t.tip_site[k] >= 0 && t.tip_site[k] < dh->nsite;
    if (!ok) { delete h; return fail(nullptr, "b200sim_create: inconsistent HandReach task", -6); }
  }
  int o = 0;
  t.st_qpos = o; o += dh->nq; t.st_qvel = o; o += dh->nv; t.st_warm = o; o += dh->nv; t.st_ctrl = o; o += dh->nu;
  t.st_mocap = o; o += 7 * dh->nmocap; t.st_pose = o; o += (t.kind == TASK_FETCH ? 7 : 0); t.st_goal = o; o += t.ngoal;
  t.st_penv = o; o += (t.penv_body > 0 ? 7 : 0);
  t.st_stride = (o + 3) & ~3;
  DevGuard guard(device);
  if (!guard.ok) { delete h; return fail(nullptr, "b200sim_create: cudaSetDevice failed", -7); }
  int nsm = 148;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device);
  h->wpb = (num_envs + nsm - 1) / nsm <= 7 ? 7 : ((num_envs + nsm - 1) / nsm <= 14 ? 14 : 28);
  h->nvp = dh->nv <= 14 ? 14 : (dh->nv == 15 ? 15 : (dh->nv <= 21 ? 21 : (dh->nv <= 30 ? 30 : (dh->nv > 32 && dh->nv <= B200_WIDE_NVP ? B200_WIDE_NVP : 0))));  // smallest built size >= nv (identity padding)
  if (h->nvp == 0) { delete h; return fail(nullptr, "b200sim_create: no kernel instantiation for this nv (31, 32 or > 36)", -8); }
  if ((t.kind == TASK_HAND || t.kind == TASK_HAND_REACH || TASK_IS_ADROIT(t.kind)) && h->nvp < 30) h->nvp = 30;  // the hand task code is compiled into this build only
  if (dh->nv <= 21 && dh->any_convex_pair) h->nvp = 22;  // arm build that carries the general convex collider (FetchSlide's puck)
  if (dh->nv <= 21 && (dh->nten > 0 || dh->nfric > 0 || dh->nsensor > 0 || dh->any_round_pair)) h->nvp = 30;  // hand features live in the NVP = 30 build
  if (h->nvp == 30 && h->wpb > 14) h->wpb = 14;  // the large models' scratch does not fit 28 envs per block
  auto fits = [&](int w) { return ((size_t)dh->hot_words + (size_t)w * dh->scr_words) * 4 + 64 <= 232448; };
  const char* ov = getenv("B200SIM_WPB");   // experiments: a block size that has no instantiation for this build is an error, not a no-op
  const int ovw = ov ? atoi(ov) : 0;
  if (h->kitchen) {
    if (dh->nv > 31) { delete h; return fail(nullptr, "b200sim_create: the kitchen build is instantiated for nv <= 31", -8); }
    h->nvp = B200_KITCHEN_NVP;
    h->wpb = h->wpb <= 7 ? 7 : ((h->kitchen_groups && fits(11)) ? 11 : (fits(10) ? 10 : 7));
    if (ov) {
      if (!((ovw == 7 || ovw == 10 || (ovw == 11 && h->kitchen_groups)) && fits(ovw))) { delete h; return fail(nullptr, "b200sim_create: B200SIM_WPB names no kitchen kernel variant that fits", -8); }
      h->wpb = ovw;
    }
  } else if (h->nvp == B200_WIDE_NVP) {
    // wide build: the largest block of {14, 13, 10, 7} warps whose scratch fits the 227 KB of shared memory (14 envs of the
    // 33-dof hammer model, 13 of the 36-dof relocate model), 7 for small batches so that every SM still gets a block
    const int want = h->wpb, cands[4] = {14, 13, 10, 7};
    h->wpb = 7;
    for (int k = 3; k >= 0; k--)
      if (cands[k] <= (want > 7 ? 14 : 7) && fits(cands[k])) h->wpb = cands[k];
    if (ov) {
      if (!((ovw == 7 || ovw == 10 || ovw == 13 || ovw == 14) && fits(ovw))) { delete h; return fail(nullptr, "b200sim_create: B200SIM_WPB names no wide kernel variant that fits", -8); }
      h->wpb = ovw;
    }
  } else if (ov) {
    if (!((ovw == 7 || ovw == 14 || (ovw == 28 && h->nvp != 30)) && fits(ovw))) { delete h; return fail(nullptr, "b200sim_create: B200SIM_WPB names no kernel variant that fits", -8); }
    h->wpb = ovw;
  }
  if (!fits(h->wpb)) { delete h; return fail(nullptr, "b200sim_create: the per-env scratch of this model does not fit the shared memory of one block", -8); }
  h->smem_bytes = ((size_t)dh->hot_words + (size_t)h->wpb * dh->scr_words) * 4;
  h->blocks = (num_envs + h->wpb - 1) / h->wpb;
  h->packed_w = (t.nobs + 2 * t.ngoal + 4 + 3) & ~3;
  cudaError_t e = cudaErrorInvalidValue;   // stays an error when no instantiation matches (wpb, nvp)
#define B200_SETATTR(W, V) if (h->wpb == W && h->nvp == V) e = cudaFuncSetAttribute(fetch_kernel<W, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes);
  B200_FOR_ALL_VARIANTS(B200_SETATTR)
#undef B200_SETATTR
  if (h->nvp == B200_WIDE_NVP) e = b200sim_wide_setattr(h->wpb, (int)h->smem_bytes) == 0 ? cudaSuccess : cudaErrorInvalidValue;
  if (h->nvp == B200_KITCHEN_NVP) e = (h->hull ? b200sim_kitchen_hull_setattr(h->wpb, (int)h->smem_bytes) : (h->kitchen_groups ? b200sim_kitchen_groups_setattr(h->wpb, (int)h->smem_bytes) : b200sim_kitchen_setattr(h->wpb, (int)h->smem_bytes))) == 0 ? cudaSuccess : cudaErrorInvalidValue;
  if (e != cudaSuccess) { std::string m = std::string("b200sim_create: no kernel variant <") + std::to_string(h->wpb) + ", " + std::to_string(h->nvp) + "> or cudaFuncSetAttribute(smem=" + std::to_string(h->smem_bytes) + ") failed: " + cudaGetErrorString(e); delete h; return fail(nullptr, m, -8); }
  const size_t state_bytes = (size_t)num_envs * t.st_stride * 4;
  if (cudaMalloc(&h->model_dev, h->model_host.size() * 4) != cudaSuccess || cudaMalloc(&h->state, state_bytes) != cudaSuccess ||
      cudaMalloc(&h->elapsed, (size_t)num_envs * 4) != cudaSuccess || cudaMalloc(&h->overflow_count, 8) != cudaSuccess) {
    free_handle(h); return fail(nullptr, "b200sim_create: cudaMalloc failed", -9);
  }
  if (cudaMemcpy(h->model_dev, h->model_host.data(), h->model_host.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemset(h->state, 0, state_bytes) != cudaSuccess || cudaMemset(h->elapsed, 0, (size_t)num_envs * 4) != cudaSuccess ||
      cudaMemset(h->overflow_count, 0, 8) != cudaSuccess) {
    free_handle(h); return fail(nullptr, "b200sim_create: uploading the model / clearing the state failed", -9);
  }
  *out = h;
  return 0;
}

void b200sim_destroy(b200sim_t* h) {
  if (!h) return;
  DevGuard guard(h->device);
  free_handle(h);
}

const char* b200sim_last_error(const b200sim_t* h) { return h ? h->err.c_str() : g_err.c_str(); }
int b200sim_num_envs(const b200sim_t* h) { return h->N; }
int b200sim_layout(const b200sim_t* h, int* out) {
  const FetchTask& t = h->task;
  out[B200SIM_ST_QPOS] = t.st_qpos; out[B200SIM_ST_QVEL] = t.st_qvel; out[B200SIM_ST_WARM] = t.st_warm; out[B200SIM_ST_CTRL] = t.st_ctrl;
  out[B200SIM_ST_MOCAP] = t.st_mocap; out[B200SIM_ST_POSE] = t.st_pose; out[B200SIM_ST_GOAL] = t.st_goal; out[B200SIM_ST_STRIDE] = t.st_stride; out[B200SIM_ST_PENV] = t.st_penv;
  return 0;
}
float* b200sim_state(b200sim_t* h) { return h->state; }
int* b200sim_elapsed(b200sim_t* h) { return h->elapsed; }
unsigned long long* b200sim_overflow_counter(b200sim_t* h) { return h->overflow_count; }
long b200sim_launch_count(const b200sim_t* h) { return h->launches; }
int b200sim_launch_config(const b200sim_t* h, int* smem_bytes, int* envs_per_block, int* blocks) {
  if (smem_bytes) *smem_bytes = (int)h->smem_bytes;
  if (envs_per_block) *envs_per_block = h->wpb;
  if (blocks) *blocks = h->blocks;
  return 0;
}
int b200sim_kernel_variant(const b200sim_t* h, int* envs_per_block, int* nvp, int* build) {
  if (envs_per_block) *envs_per_block = h->wpb;
  if (nvp) *nvp = h->nvp;
  if (build) *build = h->hull ? B200SIM_BUILD_KITCHEN_HULL : (h->kitchen ? (h->kitchen_groups ? B200SIM_BUILD_KITCHEN_GROUPS : B200SIM_BUILD_KITCHEN_FLAT)
                                                                   : (h->nvp == B200_WIDE_NVP ? B200SIM_BUILD_WIDE : B200SIM_BUILD_ARM));
  return 0;
}
int b200sim_set_time_limit(b200sim_t* h, int max_episode_steps, int terminate_on_success) {
  h->max_steps = max_episode_steps > 0 ? max_episode_steps : 0;
  h->term_on_success = terminate_on_success ? 1 : 0;
  return 0;
}
int b200sim_packed_width(const b200sim_t* h) { return h->packed_w; }
int b200sim_set_packed(b200sim_t* h, int enable) { h->packed = enable ? 1 : 0; return h->packed_w; }

static int launch(b200sim* h, int mode, int nraw, const float* actions, const unsigned char* mask, float* obs, float* achieved,
                  float* desired, float* reward, float* success, unsigned char* terminated, unsigned char* truncated, int* info, void* stream) {
  const FetchTask& t = h->task;
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.state = h->state; io.actions = actions; io.mask = mask;
  if (h->packed) {
    // one [N, W] row per env: obs | achieved | desired | reward | success | terminated | truncated (include/b200sim.h)
    if (!obs) return fail(h, "packed outputs: the `obs` argument must point at the [N, W] buffer", -1);
    io.obs = obs; io.achieved = obs + t.nobs; io.desired = io.achieved + t.ngoal; io.reward = io.desired + t.ngoal; io.success = io.reward + 1;
    io.term_f = io.reward + 2; io.trunc_f = io.reward + 3;
    io.obs_stride = io.goal_stride = io.scalar_stride = h->packed_w;
  } else {
    if (!obs || !achieved || !desired || !reward || !success) return fail(h, "output pointers must not be NULL", -1);
    io.obs = obs; io.achieved = achieved; io.desired = desired; io.reward = reward; io.success = success;
    io.obs_stride = t.nobs; io.goal_stride = t.ngoal; io.scalar_stride = 1;
  }
  io.terminated = terminated; io.truncated = truncated; io.info = info;
  io.elapsed = h->elapsed; io.max_steps = h->max_steps; io.term_on_success = h->term_on_success; io.overflow_count = h->overflow_count;
  ON_DEVICE(h);
  int matched = 0;
#define B200_LAUNCH(W, V)                                                                                   \
  if (h->wpb == W && h->nvp == V) {                                                                         \
    matched = 1;                                                                                            \
    fetch_kernel<W, V><<<h->blocks, W * 32, h->smem_bytes, (cudaStream_t)stream>>>(h->model_dev, h->task, mode, nraw, h->N, io); \
  }
  B200_FOR_ALL_VARIANTS(B200_LAUNCH)
#undef B200_LAUNCH
  if (h->nvp == B200_KITCHEN_NVP)
    matched = (h->hull ? b200sim_kitchen_hull_launch : (h->kitchen_groups ? b200sim_kitchen_groups_launch : b200sim_kitchen_launch))(h->wpb, h->blocks, h->smem_bytes, stream, h->model_dev,
                                                                                        &h->task, mode, nraw, h->N, &io) == 0;
  if (h->nvp == B200_WIDE_NVP)
    matched = b200sim_wide_launch(h->wpb, h->blocks, h->smem_bytes, stream, h->model_dev, &h->task, mode, nraw, h->N, &io) == 0;
  if (!matched) return fail(h, "no kernel variant for this (envs per block, nv) pair: nothing was launched", -8);
  h->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
#define LAUNCH_REFRESH(h, mask) launch(h, MODE_REFRESH, 0, nullptr, mask, obs, achieved, desired, reward, success, nullptr, nullptr, nullptr, stream)

int b200sim_step(b200sim_t* h, const float* actions, float* obs, float* achieved, float* desired, float* reward, float* success,
                 unsigned char* terminated, unsigned char* truncated, int* info, void* stream) {
  if (!actions) return fail(h, "b200sim_step: actions is NULL", -1);
  return launch(h, MODE_STEP, 0, actions, nullptr, obs, achieved, desired, reward, success, terminated, truncated, info, stream);
}
int b200sim_refresh(b200sim_t* h, const unsigned char* mask, float* obs, float* achieved, float* desired, float* reward,
                    float* success, void* stream) {
  return LAUNCH_REFRESH(h, mask);
}
int b200sim_reset(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_fetch_reset_t* params,
                  unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired, float* reward,
                  float* success, void* stream) {
  if (h->task.kind != TASK_FETCH) return fail(h, "b200sim_reset: the in-kernel reset draw exists for the Fetch task family only", -6);
  if (!rest_record || !params) return fail(h, "b200sim_reset: rest_record / params is NULL", -1);
  if (params->has_object && (params->obj_qadr < 0 || params->obj_qadr + 2 > h->task.st_qvel - h->task.st_qpos)) return fail(h, "b200sim_reset: obj_qadr outside qpos", -1);
  {
    ON_DEVICE(h);
    fetch_reset_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*params, seed, env_offset, h->N, mask, rest_record, h->task.st_stride,
                                                                            h->task.st_qpos, h->task.st_goal, h->state, episode, h->elapsed);
    h->launches++;
    CUDA_OK(cudaGetLastError());
  }
  return LAUNCH_REFRESH(h, mask);
}
int b200sim_reset_uniform(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_uniform_reset_t* params,
                          unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired,
                          float* reward, float* success, void* stream) {
  if (!rest_record || !params) return fail(h, "b200sim_reset_uniform: rest_record / params is NULL", -1);
  if (params->n < 0 || params->n > B200SIM_RESET_SLOTS_MAX) return fail(h, "b200sim_reset_uniform: more than 16 slots", -1);
  for (int k = 0; k < params->n; k++)
    if (params->slot[k] < -3 || params->slot[k] >= h->task.st_stride) return fail(h, "b200sim_reset_uniform: slot outside the state record", -1);
  if (params->quat_slot < -1 || params->quat_slot + 4 > h->task.st_stride) return fail(h, "b200sim_reset_uniform: quat_slot outside the state record", -1);
  {
    ON_DEVICE(h);
    uniform_reset_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*params, seed, env_offset, h->N, mask, rest_record, h->task.st_stride,
                                                                              h->state, episode, h->elapsed);
    h->launches++;
    CUDA_OK(cudaGetLastError());
  }
  return LAUNCH_REFRESH(h, mask);
}
int b200sim_reset_maze(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_maze_reset_t* params,
                       const float* goal_xy, const float* reset_xy, unsigned long long seed, int env_offset, int* episode, float* obs,
                       float* achieved, float* desired, float* reward, float* success, void* stream) {
  if (h->task.kind != TASK_ANTMAZE) return fail(h, "b200sim_reset_maze: not a maze task", -6);
  if (!rest_record || !params || !goal_xy || !reset_xy) return fail(h, "b200sim_reset_maze: NULL argument", -1);
  if (params->n_goal < 1 || params->n_reset < 1) return fail(h, "b200sim_reset_maze: empty cell table", -1);
  {
    ON_DEVICE(h);
    maze_reset_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*params, goal_xy, reset_xy, seed, env_offset, h->N, mask, rest_record,
                                                                           h->task.st_stride, h->task.st_qpos, h->task.st_goal, h->state, episode, h->elapsed);
    h->launches++;
    CUDA_OK(cudaGetLastError());
  }
  return LAUNCH_REFRESH(h, mask);
}
static int hand_reset_args(b200sim* h, const b200sim_hand_reset_t* p, const float* parallel) {
  if (h->task.kind != TASK_HAND) return fail(h, "b200sim_reset_hand_*: not a Shadow-Hand manipulation task", -6);
  if (!p || !parallel) return fail(h, "b200sim_reset_hand_*: NULL argument", -1);
  if (p->obj_qadr != h->task.obj_qadr || h->task.ngoal != 7) return fail(h, "b200sim_reset_hand_*: obj_qadr does not match the task", -1);
  if (p->rot_mode < 0 || p->rot_mode > 3 || p->goal_rot_mode < 0 || p->goal_rot_mode > 3) return fail(h, "b200sim_reset_hand_*: rot mode out of range", -1);
  return 0;
}
int b200sim_reset_hand_pose(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_hand_reset_t* params,
                            const float* parallel_quats, unsigned long long seed, int env_offset, const int* episode, int attempt,
                            void* stream) {
  if (int rc = hand_reset_args(h, params, parallel_quats)) return rc;
  if (!rest_record) return fail(h, "b200sim_reset_hand_pose: rest_record is NULL", -1);
  ON_DEVICE(h);
  hand_pose_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*params, parallel_quats, seed, env_offset, h->N, mask, rest_record,
                                                                        h->task.st_stride, h->task.st_qpos, h->task.st_goal, h->task.ngoal, h->state,
                                                                        episode, attempt);
  h->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int b200sim_reset_hand_goal(b200sim_t* h, const unsigned char* mask, const b200sim_hand_reset_t* params, const float* parallel_quats,
                            unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired,
                            float* reward, float* success, void* stream) {
  if (int rc = hand_reset_args(h, params, parallel_quats)) return rc;
  {
    ON_DEVICE(h);
    hand_goal_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*params, parallel_quats, seed, env_offset, h->N, mask, h->task.st_stride,
                                                                          h->task.st_qpos, h->task.st_goal, h->state, episode, h->elapsed);
    h->launches++;
    CUDA_OK(cudaGetLastError());
  }
  return LAUNCH_REFRESH(h, mask);
}
int b200sim_reset_reach(b200sim_t* h, const unsigned char* mask, const float* rest_record, const b200sim_reach_reset_t* params,
                        unsigned long long seed, int env_offset, int* episode, float* obs, float* achieved, float* desired, float* reward,
                        float* success, void* stream) {
  if (h->task.kind != TASK_HAND_REACH || h->task.ngoal != 15) return fail(h, "b200sim_reset_reach: not a HandReach task", -6);
  if (!rest_record || !params) return fail(h, "b200sim_reset_reach: NULL argument", -1);
  {
    ON_DEVICE(h);
    reach_reset_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*params, seed, env_offset, h->N, mask, rest_record, h->task.st_stride,
                                                                            h->task.st_goal, h->state, episode, h->elapsed);
    h->launches++;
    CUDA_OK(cudaGetLastError());
  }
  return LAUNCH_REFRESH(h, mask);
}
int b200sim_check_state(b200sim_t* h, unsigned char* bad, const float* rest_record, const b200sim_keep_t* keep, void* stream) {
  if (!bad) return fail(h, "b200sim_check_state: bad is NULL", -1);
  b200sim_keep_t k;
  k.n = 0;
  if (keep) {
    k = *keep;
    if (k.n < 0 || k.n > 4) return fail(h, "b200sim_check_state: at most 4 keep ranges", -1);
    for (int r = 0; r < k.n; r++)
      if (k.start[r] < 0 || k.len[r] < 0 || k.start[r] + k.len[r] > h->task.st_stride) return fail(h, "b200sim_check_state: keep range outside the state record", -1);
  }
  ON_DEVICE(h);
  check_state_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->N, h->task.st_stride, h->state, rest_record, k, bad);
  h->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int b200sim_raw_step_masked(b200sim_t* h, const unsigned char* mask, int nstep, float* obs, float* achieved, float* desired,
                            float* reward, float* success, void* stream) {
  return launch(h, MODE_RAW, nstep, nullptr, mask, obs, achieved, desired, reward, success, nullptr, nullptr, nullptr, stream);
}
int b200sim_raw_step(b200sim_t* h, int nstep, float* obs, float* achieved, float* desired, float* reward, float* success,
                     void* stream) {
  return launch(h, MODE_RAW, nstep, nullptr, nullptr, obs, achieved, desired, reward, success, nullptr, nullptr, nullptr, stream);
}
int b200sim_compute_reward(const b200sim_t* hc, const float* achieved, const float* desired, int M, float* out, void* stream) {
  if (M <= 0) return 0;
  b200sim* h = const_cast<b200sim*>(hc);
  ON_DEVICE(h);
  reward_kernel<<<(M + 255) / 256, 256, 0, (cudaStream_t)stream>>>(achieved, desired, M, h->task.ngoal, h->task.kind, h->task.distance_threshold,
                                                                  h->task.success_radius, h->task.reward_dense, h->task, out);
  h->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

}  // extern "C"
