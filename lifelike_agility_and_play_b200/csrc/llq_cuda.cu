// llq_cuda.cu -- host side of the sm_100a rollout engine and its C-ABI (include/llq.h).
//
// Build (see __graft_entry__.build):
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -prec-div=false -prec-sqrt=false -Xcompiler -fPIC -shared \
//        -o libllq_cuda.so llq_cuda.cu
//
// This file holds no physics: it owns device memory (structure-of-arrays state, mocap table, model constants),
// copies host buffers through pinned staging, and launches the kernels in llq_kernels.cuh.  There is no CPU
// fallback: every entry point fails with LLQ_ECUDA if the device is unusable.
#include "../../include/llq.h"
#include "../../include/llq_model_layout.h"
#include "llq_kernels.cuh"
#include "llq_step16.cuh"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

static_assert(llq::state::dim == LLQ_STATE_DIM && llq::kRecW == LLQ_ACTION_DIM + 2, "state and record layouts of include/llq.h");

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess) return fail(LLQ_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));   \
  } while (0)

constexpr int kPadFrames = 128;  // replicated tail frames so that a stale cursor never reads past the table

}  // namespace

struct llq_engine {
  llq_config cfg;
  cudaStream_t stream = nullptr;
  bool has_model = false, has_mocap = false, was_reset = false;
  // device
  llq::ModelConst* d_model = nullptr;
  llq::MocapFrame* d_frames = nullptr; int* d_clip_off = nullptr; int n_clips = 0; double frame_dt = 0; int margin = 0;
  std::vector<int> clip_off;
  llq::EnvArrays E{};
  float* d_actions = nullptr;
  int obs_dim = LLQ_OBS_DIM; bool has_init_state = false; llq::ModelConst h_model{};
  int* d_winner[2] = {nullptr, nullptr};
  double* d_avg[2] = {nullptr, nullptr};
  double* d_prob = nullptr; double* d_max_steps = nullptr;
  unsigned char* d_mask = nullptr; int* d_clip_in = nullptr; double* d_time_in = nullptr;
  double* d_ob_table = nullptr; int* d_ob_off = nullptr; bool has_obstacles = false;
  int parity = 0;
  // pinned host staging
  float* h_actions = nullptr; float* h_obs = nullptr; float* h_reward = nullptr; unsigned char* h_done = nullptr;
  void* h_scratch = nullptr; size_t h_scratch_bytes = 0;
  void* d_scratch = nullptr; size_t d_scratch_bytes = 0;
  int64_t counters[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  llq::StepParams P{};
  bool profile = false; cudaEvent_t ev[3] = {nullptr, nullptr, nullptr}; bool ev_valid = false;
  llq::SphTable* d_sph = nullptr; llq::SphTable h_sph{};   // collision spheres of the robot (llq_step16.cuh)
  int record = 0;              // "record" option: the step kernel also writes action | reward | done behind the observation of a slab row
  unsigned smem_attr_set = 0;  // bit 16 + ENV: cudaFuncAttributeMaxDynamicSharedMemorySize raised for that kernel instance on this handle's device
};

namespace {

int set_device(llq_handle h) {
  CK(cudaSetDevice(h->cfg.device));
  return LLQ_OK;
}

void fill_params(llq_handle h) {
  const llq_config& c = h->cfg;
  llq::StepParams& P = h->P;
  P.n_envs = c.n_envs; P.substeps = c.substeps; P.solver_iters = c.solver_iters;
  P.dt = (float)c.sim_dt; P.kp = (float)c.kp; P.kd = (float)c.kd; P.max_tau = (float)c.max_tau; P.gz = (float)c.gravity_z;
  P.mu = (float)(c.ground_friction * c.foot_friction);
  P.erp = (float)c.contact_erp; P.jerp = (float)c.joint_erp; P.slop = (float)c.linear_slop; P.warm = (float)c.warmstart;
  P.breaking = (float)c.contact_breaking; P.kl = (float)c.lin_damping; P.ka = (float)c.ang_damping;
  P.vmax = (float)c.max_coord_vel; P.max_imp = (float)c.max_applied_impulse;
  double sw = c.w_joint_pos + c.w_joint_vel + c.w_end_effector + c.w_root_pose + c.w_root_vel;   // PLE:365-370
  P.w_jp = (float)(c.w_joint_pos / sw); P.w_jv = (float)(c.w_joint_vel / sw); P.w_ee = (float)(c.w_end_effector / sw);
  P.w_pose = (float)(c.w_root_pose / sw); P.w_vel = (float)(c.w_root_vel / sw);
  P.sim_dt = c.sim_dt; P.frame_dt = h->frame_dt; P.margin = h->margin;
  P.max_steps = c.max_steps; P.cmd_freq_lo = c.cmd_freq_lo; P.cmd_freq_hi = c.cmd_freq_hi; P.push_start_count = c.push_start_count;
  P.push_interval = c.push_interval_steps; P.push_duration = c.push_duration_steps; P.push_enabled = c.push_enabled;
  P.mu_ground = (float)c.ground_friction; P.fr_lo = (float)c.friction_lo; P.fr_hi = (float)c.friction_hi;
  P.ph_lo = (float)c.push_h_lo; P.ph_hi = (float)c.push_h_hi; P.pv_lo = (float)c.push_v_lo; P.pv_hi = (float)c.push_v_hi;
  P.ts_lo = (float)c.target_spd_lo; P.ts_hi = (float)c.target_spd_hi;
  P.knee = c.knee_contacts; P.mu_wheel = (float)(c.ground_friction * c.link_friction); P.aux_r = (float)c.auxiliary_radius;
  P.element_id = c.element_id; P.ww_lo = (float)c.wall_width_lo; P.ww_hi = (float)c.wall_width_hi; P.wg_lo = (float)c.wall_gap_lo;
  P.wg_hi = (float)c.wall_gap_hi; P.hg_lo = (float)c.hole_gap_lo; P.hg_hi = (float)c.hole_gap_hi;
  if (!h->has_obstacles) { P.has_ob = 0; P.ob_hx = P.ob_hy = P.ob_hz = 0.f; }
}

template <typename T> int dalloc(T** p, size_t n) {
  CK(cudaMalloc((void**)p, n * sizeof(T)));
  CK(cudaMemset(*p, 0, n * sizeof(T)));
  return LLQ_OK;
}

int ensure_scratch(llq_handle h, size_t bytes) {
  if (bytes > h->h_scratch_bytes) {
    if (h->h_scratch) cudaFreeHost(h->h_scratch);
    if (h->d_scratch) cudaFree(h->d_scratch);
    h->h_scratch = nullptr; h->d_scratch = nullptr; h->h_scratch_bytes = 0;
    CK(cudaMallocHost(&h->h_scratch, bytes));
    CK(cudaMalloc(&h->d_scratch, bytes));
    h->h_scratch_bytes = h->d_scratch_bytes = bytes;
  }
  return LLQ_OK;
}

llq::MocapDev mocap_dev(llq_handle h) { return llq::MocapDev{h->d_frames, h->d_clip_off, h->n_clips, h->d_ob_table, h->d_ob_off}; }

template <int BLOCK, int ENV>
void launch_reset_t(llq_handle h, const llq::EnvArrays& E, const llq::ResetParams& RP, float* obs2, long long ld, cudaStream_t s) {
  int threads = 4 * h->cfg.n_envs;
  int grid = (threads + BLOCK - 1) / BLOCK;
  size_t smem = sizeof(double) * (size_t)(h->n_clips > 0 ? h->n_clips : 1);
  llq::pmc_reset_kernel<BLOCK, ENV><<<grid, BLOCK, smem, s>>>(E, mocap_dev(h), h->P, h->d_model, RP, obs2, ld);
}
template <int ENV>
int launch_step16(llq_handle h, const llq::EnvArrays& E, const float* a, float* obs2, long long ld, cudaStream_t s) {
  constexpr int EPB = LLQ16_BLOCK / 16;           // envs per CTA (16 lanes each)
  const int grid = (h->cfg.n_envs + EPB - 1) / EPB;
  const size_t smem = sizeof(float) * (EPB * llq::kEnvFloats + (LLQ16_BLOCK / 32) * llq::kATabWarp);
  const unsigned bit = 1u << (16 + ENV);          // static + dynamic shared memory exceeds 48 kB: per-device opt-in, once per handle
  if (!(h->smem_attr_set & bit)) {
    CK(cudaFuncSetAttribute(llq::llq_step16_kernel<ENV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    h->smem_attr_set |= bit;
  }
  llq::llq_step16_kernel<ENV><<<grid, LLQ16_BLOCK, smem, s>>>(E, mocap_dev(h), h->P, h->d_model, h->d_sph, a, obs2, ld, h->d_winner[h->parity],
                                                   (unsigned long long)h->cfg.seed, (long long)h->cfg.global_env_offset, h->record);
  return LLQ_OK;
}
int launch_step(llq_handle h, const llq::EnvArrays& E, const float* a, float* obs2, long long ld, cudaStream_t s) {
  const bool epmc = h->cfg.env_kind == LLQ_ENV_EPMC;
  h->counters[4]++;
  if (epmc && h->cfg.element_id != 0) return launch_step16<llq::kEpmcCorridor>(h, E, a, obs2, ld, s);   // the box-aware instance
  if (h->cfg.env_kind == LLQ_ENV_SEPMC) return launch_step16<llq::kSepmc>(h, E, a, obs2, ld, s);
  return epmc ? launch_step16<llq::kEpmcFlat>(h, E, a, obs2, ld, s) : launch_step16<llq::kPmc>(h, E, a, obs2, ld, s);
}
void launch_reset(llq_handle h, const llq::EnvArrays& E, const llq::ResetParams& RP, float* obs2, long long ld, cudaStream_t s) {
  if (h->cfg.env_kind == LLQ_ENV_EPMC && h->cfg.element_id != 0) launch_reset_t<128, llq::kEpmcCorridor>(h, E, RP, obs2, ld, s);
  else if (h->cfg.env_kind == LLQ_ENV_EPMC) launch_reset_t<128, llq::kEpmcFlat>(h, E, RP, obs2, ld, s);
  else if (h->cfg.env_kind == LLQ_ENV_SEPMC) launch_reset_t<128, llq::kSepmc>(h, E, RP, obs2, ld, s);
  else launch_reset_t<128, llq::kPmc>(h, E, RP, obs2, ld, s);
  h->counters[4]++;
}

llq::ResetParams reset_params(llq_handle h, int mode, bool update_table) {
  llq::ResetParams RP{};
  RP.mode = mode; RP.mask = nullptr; RP.clip_in = nullptr; RP.time_in = nullptr;
  RP.seed = h->cfg.seed; RP.gid0 = h->cfg.global_env_offset;
  RP.winner_cur = h->d_winner[h->parity]; RP.winner_next = h->d_winner[h->parity ^ 1];
  RP.avg_old = h->d_avg[h->parity]; RP.avg_new = update_table ? h->d_avg[h->parity ^ 1] : h->d_avg[h->parity];
  RP.prob = h->d_prob; RP.max_steps = h->d_max_steps; RP.factor = h->cfg.prioritized_sample_factor;
  RP.update_table = update_table ? 1 : 0;
  return RP;
}

int check_ready(llq_handle h, bool need_reset) {
  if (!h) return fail(LLQ_EINVAL, "null handle");
  if (!h->has_model) return fail(LLQ_ESTATE, "llq_load_model has not been called");
  if (h->cfg.env_kind == LLQ_ENV_PMC && !h->has_mocap) return fail(LLQ_ESTATE, "llq_load_mocap has not been called");
  if (h->cfg.env_kind != LLQ_ENV_PMC && !h->has_init_state) return fail(LLQ_ESTATE, "llq_set_init_state has not been called");
  if (need_reset && !h->was_reset) return fail(LLQ_ESTATE, "llq_reset has not been called");
  return set_device(h);
}

void copy_item(llq::DampItem& d, const double* s) {
  d.m = (float)s[0];
  for (int i = 0; i < 3; i++) d.c[i] = (float)s[1 + i];
  for (int i = 0; i < 6; i++) d.Ic[i] = (float)s[4 + i];
}

// SoA <-> AoS helpers for the state field (host side, after a D2H of the raw arrays)
int get_soa_f(llq_handle h, const float* d_src, int width, float* dst) {
  const int n = h->cfg.n_envs;
  int rc = ensure_scratch(h, sizeof(float) * (size_t)width * n);
  if (rc) return rc;
  CK(cudaMemcpyAsync(h->h_scratch, d_src, sizeof(float) * (size_t)width * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  const float* s = (const float*)h->h_scratch;
  for (int i = 0; i < n; i++)
    for (int t = 0; t < width; t++) dst[(size_t)i * width + t] = s[(size_t)t * n + i];
  return LLQ_OK;
}

}  // namespace

extern "C" {

int llq_abi_version(int* is_cuda) {
  if (is_cuda) *is_cuda = 1;
  return LLQ_ABI_VERSION;
}

int llq_default_config(llq_config* c) {
  if (!c) return fail(LLQ_EINVAL, "null config");
  std::memset(c, 0, sizeof(*c));
  c->struct_size = (int32_t)sizeof(llq_config);
  c->n_envs = 1; c->device = 0; c->substeps = 10; c->solver_iters = 10; c->auto_reset = 0; c->num_threads = 0;
  c->global_env_offset = 0; c->seed = 0;
  c->sim_dt = 1.0 / 500.0; c->policy_dt = 1.0 / 50.0;
  c->kp = 50.0; c->kd = 0.5; c->max_tau = 18.0;
  c->gravity_z = -9.80665; c->ground_friction = 0.9; c->foot_friction = 0.5;
  c->contact_erp = 0.08; c->joint_erp = 0.2; c->linear_slop = 1e-5; c->warmstart = 0.1;
  c->contact_breaking = 0.02 * 0.025;
  c->lin_damping = 0.04; c->ang_damping = 0.04; c->max_coord_vel = 100.0; c->max_applied_impulse = 1000.0;
  c->w_joint_pos = 0.3; c->w_joint_vel = 0.05; c->w_end_effector = 0.1; c->w_root_pose = 0.5; c->w_root_vel = 0.05;
  c->prioritized_sample_factor = 3.0;
  // EPMC defaults = train_scripts/example_epmc_train.sh:100-117 (only used when env_kind = LLQ_ENV_EPMC)
  c->env_kind = LLQ_ENV_PMC; c->max_steps = 1000; c->cmd_freq_lo = 9999; c->cmd_freq_hi = 10000;
  c->push_start_count = -250; c->push_interval_steps = 499; c->push_duration_steps = 100; c->push_enabled = 1;
  c->friction_lo = 0.4; c->friction_hi = 3.0; c->push_h_lo = 0.0; c->push_h_hi = 50.0; c->push_v_lo = 0.0; c->push_v_hi = 10.0;
  c->target_spd_lo = 0.5; c->target_spd_hi = 3.0;
  c->element_id = 0; c->wall_width_lo = 0.02; c->wall_width_hi = 0.5; c->wall_gap_lo = 1.0; c->wall_gap_hi = 20.0;
  c->hole_gap_lo = 0.25; c->hole_gap_hi = 0.3;
  c->knee_contacts = 2; c->reserved1 = 0; c->link_friction = 0.5; c->auxiliary_radius = 0.0;
  return LLQ_OK;
}

int llq_create(const llq_config* cfg, llq_handle* out) {
  if (!cfg || !out) return fail(LLQ_EINVAL, "null argument");
  if (cfg->struct_size != (int32_t)sizeof(llq_config)) return fail(LLQ_EINVAL, "llq_config size mismatch (ABI)");
  if (cfg->n_envs <= 0) return fail(LLQ_EINVAL, "n_envs must be positive");
  if (cfg->substeps <= 0 || cfg->solver_iters < 0 || !(cfg->sim_dt > 0)) return fail(LLQ_EINVAL, "bad step configuration");
  if (cfg->env_kind != LLQ_ENV_PMC && cfg->env_kind != LLQ_ENV_EPMC && cfg->env_kind != LLQ_ENV_SEPMC) return fail(LLQ_EINVAL, "unknown env_kind");
  if (cfg->env_kind == LLQ_ENV_SEPMC && (cfg->n_envs % 2 != 0 || cfg->max_steps <= 0 || cfg->push_interval_steps <= 0))
    return fail(LLQ_EINVAL, "SEPMC: n_envs counts robots and must be even");
  if (cfg->env_kind == LLQ_ENV_EPMC && (cfg->max_steps <= 0 || cfg->cmd_freq_hi <= cfg->cmd_freq_lo || cfg->cmd_freq_lo <= 0 ||
                                        cfg->push_interval_steps <= 0))
    return fail(LLQ_EINVAL, "bad EPMC configuration");
  if (cfg->env_kind == LLQ_ENV_EPMC && (cfg->element_id < 0 || cfg->element_id > 3)) return fail(LLQ_EINVAL, "EPMC element_id must be 0..3");
  if (cfg->knee_contacts < 0 || cfg->knee_contacts > 2) return fail(LLQ_EINVAL, "knee_contacts must be 0, 1 or 2");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(LLQ_ECUDA, "no CUDA device visible (the CUDA engine has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(LLQ_EINVAL, "device ordinal out of range");
  llq_engine* h = new (std::nothrow) llq_engine();
  if (!h) return fail(LLQ_ENOMEM, "out of memory");
  h->cfg = *cfg;
  h->obs_dim = cfg->env_kind == LLQ_ENV_EPMC ? LLQ_OBS_DIM_EPMC : (cfg->env_kind == LLQ_ENV_SEPMC ? LLQ_OBS_DIM_SEPMC : LLQ_OBS_DIM);
  int rc = set_device(h);
  if (rc) { delete h; return rc; }
  const size_t n = (size_t)cfg->n_envs;
#define TRY(x) do { rc = (x); if (rc) { llq_destroy(h); return rc; } } while (0)
  cudaError_t ce = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (ce != cudaSuccess) { delete h; return fail(LLQ_ECUDA, cudaGetErrorString(ce)); }
  TRY(dalloc(&h->d_model, 1)); TRY(dalloc(&h->d_sph, 1));
  TRY(dalloc(&h->E.pos, 3 * n)); TRY(dalloc(&h->E.st, llq::st::dim * n)); TRY(dalloc(&h->E.time, n)); TRY(dalloc(&h->E.clip, n));
  TRY(dalloc(&h->E.reward_sum, n)); TRY(dalloc(&h->E.episode_steps, n)); TRY(dalloc(&h->E.episode, n));
  TRY(dalloc(&h->E.warm, LLQ_MAX_SPHERES * n)); TRY(dalloc(&h->E.obs, (size_t)h->obs_dim * n)); TRY(dalloc(&h->E.kin, llq::state::dim * n));
  TRY(dalloc(&h->E.foot_pos, 12 * n)); TRY(dalloc(&h->E.done_reward, n)); TRY(dalloc(&h->E.done, n)); TRY(dalloc(&h->E.reward, n));
  TRY(dalloc(&h->E.counters, 8));
  TRY(dalloc(&h->E.aux, (size_t)LLQ_AUX_DIM * n));
  TRY(dalloc(&h->E.ob_id, n));
  TRY(dalloc(&h->E.boxes, (size_t)6 * LLQ_MAX_BOXES * n)); TRY(dalloc(&h->E.nbox, n));
  TRY(dalloc(&h->d_actions, (size_t)LLQ_ACTION_DIM * n));
  TRY(dalloc(&h->d_mask, n)); TRY(dalloc(&h->d_clip_in, n)); TRY(dalloc(&h->d_time_in, n));
  ce = cudaMallocHost((void**)&h->h_actions, sizeof(float) * LLQ_ACTION_DIM * n);
  if (ce == cudaSuccess) ce = cudaMallocHost((void**)&h->h_obs, sizeof(float) * h->obs_dim * n);
  if (ce == cudaSuccess) ce = cudaMallocHost((void**)&h->h_reward, sizeof(float) * n);
  if (ce == cudaSuccess) ce = cudaMallocHost((void**)&h->h_done, n);
  if (ce != cudaSuccess) { llq_destroy(h); return fail(LLQ_ECUDA, cudaGetErrorString(ce)); }
#undef TRY
  if (cfg->env_kind != LLQ_ENV_PMC) {   // no mocap table: the winner/avg buffers are still passed to the kernels (unused)
    h->frame_dt = 1.0 / 120.0; h->margin = 0;
    fill_params(h);
  }
  *out = h;
  return LLQ_OK;
}

int llq_destroy(llq_handle h) {
  if (!h) return LLQ_OK;
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  void* dptrs[] = {h->d_sph, h->d_model, h->d_frames, h->d_clip_off, h->E.pos, h->E.st, h->E.time, h->E.clip, h->E.reward_sum, h->E.episode_steps,
                   h->E.episode, h->E.warm, h->E.obs, h->E.kin, h->E.foot_pos, h->E.done_reward, h->E.done, h->E.reward, h->E.counters, h->E.aux, h->E.ob_id, h->E.boxes, h->E.nbox, h->d_ob_table, h->d_ob_off,
                   h->d_actions, h->d_winner[0], h->d_winner[1], h->d_avg[0], h->d_avg[1], h->d_prob, h->d_max_steps, h->d_mask,
                   h->d_clip_in, h->d_time_in, h->d_scratch};
  for (void* p : dptrs) if (p) cudaFree(p);
  void* hptrs[] = {h->h_actions, h->h_obs, h->h_reward, h->h_done, h->h_scratch};
  for (void* p : hptrs) if (p) cudaFreeHost(p);
  for (int i = 0; i < 3; i++) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return LLQ_OK;
}

int llq_load_model(llq_handle h, const double* b, int64_t n) {
  if (!h || !b) return fail(LLQ_EINVAL, "null argument");
  if (n < LLQ_HDR || (int64_t)b[LLQ_H_MAGIC] != LLQ_MODEL_MAGIC || (int64_t)b[LLQ_H_TOTAL] != n)
    return fail(LLQ_EINVAL, "bad model blob (magic/size)");
  if ((int)b[LLQ_H_NDOF] != 12) return fail(LLQ_EUNSUPPORTED, "engine expects 12 actuated joints");
  int rc = set_device(h);
  if (rc) return rc;
  const double* sp = b + (int64_t)b[LLQ_H_OFF_SPECIAL];
  llq::ModelConst M;
  std::memset(&M, 0, sizeof(M));
  for (int i = 0; i < 4; i++) M.base.qI[i] = (float)sp[LLQ_S_QI + i];
  M.base.m = (float)sp[LLQ_S_BASE_M];
  for (int i = 0; i < 3; i++) M.base.h[i] = (float)sp[LLQ_S_BASE_H + i];
  for (int i = 0; i < 6; i++) M.base.I[i] = (float)sp[LLQ_S_BASE_I + i];
  M.base.nd = (int)sp[LLQ_S_BASE_ND];
  if (M.base.nd < 0 || M.base.nd > 3) return fail(LLQ_EINVAL, "bad base damping item count");
  for (int t = 0; t < M.base.nd; t++) copy_item(M.base.d[t], sp + LLQ_S_BASE_DAMP + t * LLQ_DAMP_ITEM);
  static const int want_axis[3] = {0, 1, 1};
  static const int want_sign[3] = {1, -1, -1};
  for (int k = 0; k < 4; k++) {
    const double* lb = sp + LLQ_S_LEGS + k * LLQ_LEG;
    for (int j = 0; j < 3; j++) {
      const double* jb = lb + j * LLQ_LJ;
      llq::JointConst& J = M.leg[k].j[j];
      if ((int)jb[LLQ_J_AXIS_IDX] != want_axis[j] || (int)jb[LLQ_J_AXIS_SIGN] != want_sign[j])
        return fail(LLQ_EUNSUPPORTED, "kernel is specialised for hip:+x, thigh:-y, shank:-y joint axes (max.urdf)");
      for (int i = 0; i < 3; i++) { J.r[i] = (float)jb[LLQ_J_R + i]; J.h[i] = (float)jb[LLQ_J_H + i]; }
      J.m = (float)jb[LLQ_J_M];
      for (int i = 0; i < 6; i++) J.I[i] = (float)jb[LLQ_J_I + i];
      J.nd = (int)jb[LLQ_J_ND];
      if (J.nd < 0 || J.nd > 2) return fail(LLQ_EINVAL, "bad joint damping item count");
      for (int t = 0; t < J.nd; t++) copy_item(J.d[t], jb + LLQ_J_DAMP + t * LLQ_DAMP_ITEM);
      J.lower = (float)jb[LLQ_J_LOWER]; J.upper = (float)jb[LLQ_J_UPPER]; J.haslim = jb[LLQ_J_HASLIM] != 0; J.jdamp = (float)jb[LLQ_J_JDAMP];
    }
    for (int i = 0; i < 3; i++) M.leg[k].foot[i] = (float)lb[LLQ_L_FOOT + i];
    M.leg[k].foot_r = (float)lb[LLQ_L_FOOT + 3];
  }
  {   // FR hip = generic link 1: inertial-frame rotation and CoM (for the EPMC push force)
    const double* g = b + (int64_t)b[LLQ_H_OFF_GENERIC] + 1 * LLQ_GL;
    for (int i = 0; i < 9; i++) M.push_R[i] = (float)g[LLQ_G_RIN + i];
    for (int i = 0; i < 3; i++) M.push_c[i] = (float)g[LLQ_G_COM + i];
  }
  {   // detection proxies for the hurdle plate
    const double* pr = b + (int64_t)b[LLQ_H_OFF_PROXIES];
    const double* gen = b + (int64_t)b[LLQ_H_OFF_GENERIC];
    int nw = 0, nh = 0, nc = 0, nhd = 0;
    for (int i = 0; i < (int)b[LLQ_H_NPROXIES]; i++, pr += LLQ_PROXY) {
      const int link = (int)pr[0], kind = (int)pr[5];
      if (kind == 4 && nhd < 2) {         // handle (fixed to the body): joint origin + shape offset, relative to the base reference point
        const double* g = gen + (size_t)link * LLQ_GL;
        for (int t = 0; t < 3; t++) M.handle[nhd][t] = (float)(g[LLQ_G_JXYZ + t] + pr[1 + t] - gen[LLQ_G_COM + t]);
        M.handle[nhd++][3] = (float)pr[4];
      }
      if (kind == 1 && nw < 4) {          // wheel: its (fixed) joint origin in the thigh frame + the shape offset (joint rpy only spins the symmetric cylinder)
        const double* g = gen + (size_t)link * LLQ_GL;
        for (int t = 0; t < 3; t++) M.wheel_off[nw][t] = (float)(g[LLQ_G_JXYZ + t] + pr[1 + t]);
        M.wheel_r[nw++] = (float)pr[4];
      } else if (kind == 2 && nh < 4) {
        M.hip_r[nh++] = (float)pr[4];
      } else if (kind == 3 && nc < 8) {   // body corner, relative to the base reference point (body CoM), body axes
        const double* g0 = gen;
        for (int t = 0; t < 3; t++) M.corner[nc][t] = (float)(pr[1 + t] - g0[LLQ_G_COM + t]);
        nc++;
      }
    }
    if ((int)b[LLQ_H_NPROXIES] > 0 && (nw != 4 || nh != 4 || nc != 8)) return fail(LLQ_EINVAL, "unexpected proxy table");
  }
  {   // collision spheres (llq_step16.cuh): centre in the frame of the articulated link they ride on
    llq::SphTable& T = h->h_sph;
    std::memset(&T, 0, sizeof(T));
    T.rule = h->cfg.knee_contacts;
    const double* sps = b + (int64_t)b[LLQ_H_OFF_SPHERES];
    const double* gen = b + (int64_t)b[LLQ_H_OFF_GENERIC];
    const int ns = (int)b[LLQ_H_NSPHERES];
    int nfoot = 0;
    for (int i = 0; i < ns; i++, sps += LLQ_SPH) {
      const int kind = (int)sps[6];
      if (kind != 0 && !(T.rule == 2 || (T.rule == 1 && kind == 1))) continue;
      if (T.n >= llq::kMaxSph) return fail(LLQ_EINVAL, "too many collision spheres");
      llq::SphConst& S = T.s[T.n++];
      if (kind == 0) {            // foot k: its centre in the shank frame comes from the special section
        if (nfoot >= 4) return fail(LLQ_EINVAL, "more than four foot spheres");
        for (int t = 0; t < 3; t++) S.c[t] = M.leg[nfoot].foot[t];
        S.r = M.leg[nfoot].foot_r; S.leg = nfoot; S.depth = 3; S.foot = 1; S.mu_link = 0.f;
        nfoot++;
        continue;
      }
      const int link = (int)sps[0];
      const double* g = gen + (size_t)link * LLQ_GL;
      S.r = (float)sps[4]; S.foot = 0; S.mu_link = (float)(h->cfg.ground_friction * h->cfg.link_friction);
      if (link == 0) {            // trunk: relative to the base reference point (body CoM), body axes
        S.leg = 0; S.depth = 0;
        for (int t = 0; t < 3; t++) S.c[t] = (float)(sps[1 + t] - gen[LLQ_G_COM + t]);
      } else {
        if ((int)g[LLQ_G_JTYPE] != 1) return fail(LLQ_EINVAL, "collision spheres must ride on the base or on an actuated link");
        const int dof = (int)g[LLQ_G_DOF];
        S.leg = dof / 3; S.depth = dof % 3 + 1;
        for (int t = 0; t < 3; t++) S.c[t] = (float)sps[1 + t];
      }
    }
    if (nfoot != 4) return fail(LLQ_EINVAL, "model blob must list the four foot spheres first");
    CK(cudaMemcpy(h->d_sph, &T, sizeof(T), cudaMemcpyHostToDevice));
  }
  for (int i = 0; i < llq::state::dim; i++) M.init_state[i] = h->h_model.init_state[i];
  h->h_model = M;
  CK(cudaMemcpy(h->d_model, &M, sizeof(M), cudaMemcpyHostToDevice));
  h->has_model = true;
  return LLQ_OK;
}

int llq_obs_dim(llq_handle h) { return h ? h->obs_dim : fail(LLQ_EINVAL, "null handle"); }

int llq_set_init_state(llq_handle h, const double* st) {
  if (!h || !st) return fail(LLQ_EINVAL, "null argument");
  int rc = set_device(h);
  if (rc) return rc;
  for (int i = 0; i < llq::state::dim; i++) h->h_model.init_state[i] = (float)st[i];
  if (h->has_model) CK(cudaMemcpy(h->d_model, &h->h_model, sizeof(h->h_model), cudaMemcpyHostToDevice));
  h->has_init_state = true;
  return LLQ_OK;
}

int llq_load_mocap(llq_handle h, const double* frames, const int32_t* off, int32_t n_clips, double frame_dt) {
  if (!h || !frames || !off || n_clips <= 0 || !(frame_dt > 0)) return fail(LLQ_EINVAL, "bad mocap arguments");
  int rc = set_device(h);
  if (rc) return rc;
  h->frame_dt = frame_dt;
  int frame_rate = (int)(1.0 / frame_dt);                                                     // ML:34
  h->margin = (int)std::ceil(h->cfg.policy_dt / frame_dt) + frame_rate + 2;                   // ML:35
  for (int c = 0; c < n_clips; c++)
    if (off[c + 1] - off[c] < h->margin + 3) return fail(LLQ_EINVAL, "mocap clip shorter than margin + 3 frames");
  h->n_clips = n_clips;
  h->clip_off.assign(off, off + n_clips + 1);
  const size_t total = (size_t)off[n_clips];
  std::vector<llq::MocapFrame> tab(total + kPadFrames);
  for (size_t f = 0; f < total + kPadFrames; f++) {
    const double* s = frames + std::min(f, total - 1) * LLQ_MOCAP_FRAME;
    llq::MocapFrame& d = tab[f];
    d.x = s[0]; d.y = s[1]; d.z = s[2]; d.pad = 0;
    for (int i = 0; i < 4; i++) d.quat[i] = (float)s[3 + i];
    for (int i = 0; i < 12; i++) d.q[i] = (float)s[7 + i];
  }
  void* olds[] = {h->d_frames, h->d_clip_off, h->d_winner[0], h->d_winner[1], h->d_avg[0], h->d_avg[1], h->d_prob, h->d_max_steps};
  for (void* p : olds) if (p) cudaFree(p);
  h->d_frames = nullptr;
  CK(cudaMalloc((void**)&h->d_frames, tab.size() * sizeof(llq::MocapFrame)));
  CK(cudaMemcpy(h->d_frames, tab.data(), tab.size() * sizeof(llq::MocapFrame), cudaMemcpyHostToDevice));
  CK(cudaMalloc((void**)&h->d_clip_off, sizeof(int) * (n_clips + 1)));
  CK(cudaMemcpy(h->d_clip_off, off, sizeof(int) * (n_clips + 1), cudaMemcpyHostToDevice));
  std::vector<int> neg(n_clips, -1);
  std::vector<double> ms(n_clips), zeros(n_clips, 0.0), pr(n_clips, 1.0 / n_clips);
  for (int c = 0; c < n_clips; c++) ms[c] = (off[c + 1] - off[c] - h->margin) * frame_dt / h->cfg.policy_dt;   // ML:45
  for (int p = 0; p < 2; p++) {
    CK(cudaMalloc((void**)&h->d_winner[p], sizeof(int) * n_clips));
    CK(cudaMemcpy(h->d_winner[p], neg.data(), sizeof(int) * n_clips, cudaMemcpyHostToDevice));
    CK(cudaMalloc((void**)&h->d_avg[p], sizeof(double) * n_clips));
    CK(cudaMemcpy(h->d_avg[p], zeros.data(), sizeof(double) * n_clips, cudaMemcpyHostToDevice));
  }
  CK(cudaMalloc((void**)&h->d_prob, sizeof(double) * n_clips));
  CK(cudaMemcpy(h->d_prob, pr.data(), sizeof(double) * n_clips, cudaMemcpyHostToDevice));
  CK(cudaMalloc((void**)&h->d_max_steps, sizeof(double) * n_clips));
  CK(cudaMemcpy(h->d_max_steps, ms.data(), sizeof(double) * n_clips, cudaMemcpyHostToDevice));
  h->parity = 0;
  h->has_mocap = true;
  fill_params(h);
  return LLQ_OK;
}

int llq_load_obstacles(llq_handle h, const double* table, const int32_t* offsets, int32_t n_clips, double hx, double hy, double hz) {
  if (!h || !offsets || n_clips <= 0) return fail(LLQ_EINVAL, "bad obstacle arguments");
  if (!h->has_mocap || n_clips != h->n_clips) return fail(LLQ_ESTATE, "llq_load_obstacles needs the mocap table first (same clip count)");
  if (offsets[0] != 0 || (offsets[n_clips] > 0 && !table)) return fail(LLQ_EINVAL, "bad obstacle table");
  for (int c = 0; c < n_clips; c++) if (offsets[c + 1] < offsets[c]) return fail(LLQ_EINVAL, "obstacle offsets must be non-decreasing");
  int rc = set_device(h);
  if (rc) return rc;
  if (h->d_ob_table) cudaFree(h->d_ob_table);
  if (h->d_ob_off) cudaFree(h->d_ob_off);
  h->d_ob_table = nullptr; h->d_ob_off = nullptr;
  const size_t total = (size_t)offsets[n_clips];
  CK(cudaMalloc((void**)&h->d_ob_table, sizeof(double) * 4 * (total ? total : 1)));
  if (total) CK(cudaMemcpy(h->d_ob_table, table, sizeof(double) * 4 * total, cudaMemcpyHostToDevice));
  CK(cudaMalloc((void**)&h->d_ob_off, sizeof(int) * (n_clips + 1)));
  CK(cudaMemcpy(h->d_ob_off, offsets, sizeof(int) * (n_clips + 1), cudaMemcpyHostToDevice));
  h->has_obstacles = true;
  h->P.has_ob = 1; h->P.ob_hx = (float)hx; h->P.ob_hy = (float)hy; h->P.ob_hz = (float)hz;
  return LLQ_OK;
}

static int do_reset(llq_handle h, const uint8_t* mask, const int32_t* clip, const double* time, float* obs) {
  const size_t n = (size_t)h->cfg.n_envs;
  llq::ResetParams RP = reset_params(h, clip ? 2 : 1, false);
  if (mask) {
    std::memcpy(h->h_done, mask, n);   // reuse the pinned done buffer as the mask staging area
    CK(cudaMemcpyAsync(h->d_mask, h->h_done, n, cudaMemcpyHostToDevice, h->stream));
    RP.mask = h->d_mask;
  }
  if (clip) {
    for (size_t i = 0; i < n; i++) {
      if (mask && !mask[i]) continue;
      if (clip[i] < 0 || clip[i] >= h->n_clips) return fail(LLQ_EINVAL, "clip id out of range");
      int nf = h->clip_off[clip[i] + 1] - h->clip_off[clip[i]];
      if (!(time[i] >= 0) || time[i] >= h->frame_dt * (nf - h->margin - 1)) return fail(LLQ_EINVAL, "reset time outside clip");
    }
    int rc = ensure_scratch(h, n * (sizeof(int) + sizeof(double)));
    if (rc) return rc;
    double* ht = (double*)h->h_scratch; int* hc = (int*)(ht + n);
    std::memcpy(ht, time, n * sizeof(double)); std::memcpy(hc, clip, n * sizeof(int));
    CK(cudaMemcpyAsync(h->d_time_in, ht, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_clip_in, hc, n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    RP.clip_in = h->d_clip_in; RP.time_in = h->d_time_in;
  }
  launch_reset(h, h->E, RP, nullptr, h->obs_dim, h->stream);
  CK(cudaGetLastError());
  if (obs) CK(cudaMemcpyAsync(h->h_obs, h->E.obs, sizeof(float) * h->obs_dim * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (obs) std::memcpy(obs, h->h_obs, sizeof(float) * h->obs_dim * n);
  h->was_reset = true;
  return LLQ_OK;
}

int llq_reset(llq_handle h, const uint8_t* mask, float* obs) {
  int rc = check_ready(h, false);
  if (rc) return rc;
  return do_reset(h, mask, nullptr, nullptr, obs);
}

int llq_reset_to(llq_handle h, const uint8_t* mask, const int32_t* clip, const double* time, float* obs) {
  int rc = check_ready(h, false);
  if (rc) return rc;
  if (h->cfg.env_kind != LLQ_ENV_PMC) return fail(LLQ_EUNSUPPORTED, "llq_reset_to is a PMC (mocap) entry point");
  if (!clip || !time) return fail(LLQ_EINVAL, "null clip/time");
  return do_reset(h, mask, clip, time, obs);
}

int llq_step_ex(llq_handle h, const float* actions, float* obs, int64_t obs_ld, float* reward, uint8_t* done, int io_mode,
                void* stream) {
  int rc = check_ready(h, true);
  if (rc) return rc;
  if (!actions) return fail(LLQ_EINVAL, "null actions");
  const size_t od = (size_t)h->obs_dim;
  if (obs && obs_ld < (int64_t)od) return fail(LLQ_EINVAL, "obs_ld smaller than the observation width");
  if (h->record && io_mode == LLQ_IO_DEVICE && obs && obs_ld < (int64_t)od + llq::kRecW)
    return fail(LLQ_EINVAL, "record mode needs obs_ld >= observation width + " + std::to_string(llq::kRecW) + " (action | reward | done)");
  const size_t n = (size_t)h->cfg.n_envs;
  llq::EnvArrays E = h->E;
  const float* d_act;
  float* obs2 = nullptr;
  cudaStream_t s = h->stream;
  if (io_mode == LLQ_IO_DEVICE) {
    if (stream) s = (cudaStream_t)stream;
    d_act = actions;
    if (reward) E.reward = reward;
    if (done) E.done = done;
    obs2 = obs;
  } else if (io_mode == LLQ_IO_HOST) {
    std::memcpy(h->h_actions, actions, sizeof(float) * LLQ_ACTION_DIM * n);
    CK(cudaMemcpyAsync(h->d_actions, h->h_actions, sizeof(float) * LLQ_ACTION_DIM * n, cudaMemcpyHostToDevice, s));
    d_act = h->d_actions;
  } else if (io_mode == LLQ_IO_PINNED) {
    CK(cudaMemcpyAsync(h->d_actions, actions, sizeof(float) * LLQ_ACTION_DIM * n, cudaMemcpyHostToDevice, s));
    d_act = h->d_actions;
  } else {
    return fail(LLQ_EINVAL, "bad io_mode");
  }
  if (h->profile) CK(cudaEventRecord(h->ev[0], s));
  rc = launch_step(h, E, d_act, obs2, (long long)obs_ld, s);
  if (rc) return rc;
  if (h->profile) CK(cudaEventRecord(h->ev[1], s));
  // prioritized-sampling table update (PLE:235-240) + auto reset of finished envs
  llq::ResetParams RP = reset_params(h, h->cfg.auto_reset ? 0 : 3, true);
  launch_reset(h, E, RP, obs2, (long long)obs_ld, s);
  if (h->profile) { CK(cudaEventRecord(h->ev[2], s)); h->ev_valid = true; }
  h->parity ^= 1;
  CK(cudaGetLastError());
  h->counters[0] += (int64_t)n;
  if (io_mode == LLQ_IO_HOST) {
    if (obs) CK(cudaMemcpyAsync(h->h_obs, h->E.obs, sizeof(float) * od * n, cudaMemcpyDeviceToHost, s));
    if (reward) CK(cudaMemcpyAsync(h->h_reward, h->E.reward, sizeof(float) * n, cudaMemcpyDeviceToHost, s));
    if (done) CK(cudaMemcpyAsync(h->h_done, h->E.done, n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (obs) {
      if ((size_t)obs_ld == od) std::memcpy(obs, h->h_obs, sizeof(float) * od * n);
      else for (size_t i = 0; i < n; i++) std::memcpy(obs + i * obs_ld, h->h_obs + i * od, sizeof(float) * od);
    }
    if (reward) std::memcpy(reward, h->h_reward, sizeof(float) * n);
    if (done) std::memcpy(done, h->h_done, n);
  } else if (io_mode == LLQ_IO_PINNED) {
    if (obs) {
      if ((size_t)obs_ld == od) CK(cudaMemcpyAsync(obs, h->E.obs, sizeof(float) * od * n, cudaMemcpyDeviceToHost, s));
      else CK(cudaMemcpy2DAsync(obs, sizeof(float) * obs_ld, h->E.obs, sizeof(float) * od, sizeof(float) * od, n, cudaMemcpyDeviceToHost, s));
    }
    if (reward) CK(cudaMemcpyAsync(reward, h->E.reward, sizeof(float) * n, cudaMemcpyDeviceToHost, s));
    if (done) CK(cudaMemcpyAsync(done, h->E.done, n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  return LLQ_OK;
}

int llq_step(llq_handle h, const float* actions, float* obs, float* reward, uint8_t* done) {
  if (!h) return fail(LLQ_EINVAL, "null handle");
  return llq_step_ex(h, actions, obs, h->obs_dim, reward, done, LLQ_IO_HOST, nullptr);
}

int llq_get_field(llq_handle h, int field, void* dst) {
  if (!h || !dst) return fail(LLQ_EINVAL, "null argument");
  int rc = set_device(h);
  if (rc) return rc;
  const size_t n = (size_t)h->cfg.n_envs;
  CK(cudaStreamSynchronize(h->stream));
  switch (field) {
    case LLQ_F_STATE: {
      std::vector<float> tmp(llq::st::dim * n);
      rc = get_soa_f(h, h->E.st, llq::st::dim, tmp.data());
      if (rc) return rc;
      std::vector<double> pos(3 * n);
      CK(cudaMemcpy(pos.data(), h->E.pos, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost));
      float* o = (float*)dst;
      for (size_t i = 0; i < n; i++) {
        for (int t = 0; t < 3; t++) o[i * llq::state::dim + llq::state::pos + t] = (float)pos[t * n + i];
        for (int t = 0; t < llq::st::dim; t++) o[i * llq::state::dim + llq::state::quat + t] = tmp[i * llq::st::dim + t];
      }
      return LLQ_OK;
    }
    case LLQ_F_KIN_STATE: return get_soa_f(h, h->E.kin, llq::state::dim, (float*)dst);
    case LLQ_F_WARMSTART: return get_soa_f(h, h->E.warm, LLQ_MAX_SPHERES, (float*)dst);
    case LLQ_F_FOOT_POS: return get_soa_f(h, h->E.foot_pos, 12, (float*)dst);
    case LLQ_F_CLIP: CK(cudaMemcpy(dst, h->E.clip, sizeof(int) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_TIME: CK(cudaMemcpy(dst, h->E.time, sizeof(double) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_REWARD_SUM: CK(cudaMemcpy(dst, h->E.reward_sum, sizeof(float) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_EPISODE_STEPS: CK(cudaMemcpy(dst, h->E.episode_steps, sizeof(int) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_EPISODE_ID: CK(cudaMemcpy(dst, h->E.episode, sizeof(long long) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_OB_ID: CK(cudaMemcpy(dst, h->E.ob_id, sizeof(int) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_OBS: CK(cudaMemcpy(dst, h->E.obs, sizeof(float) * h->obs_dim * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_BOXES: {
      std::vector<int> nb(n);
      CK(cudaMemcpy(dst, h->E.boxes, sizeof(float) * 6 * LLQ_MAX_BOXES * n, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(nb.data(), h->E.nbox, sizeof(int) * n, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < n; i++)                      // rows past the env's box count hold stale boxes of earlier episodes
        for (int b = nb[i]; b < LLQ_MAX_BOXES; b++) std::memset((float*)dst + (i * LLQ_MAX_BOXES + b) * 6, 0, 6 * sizeof(float));
      return LLQ_OK;
    }
    case LLQ_F_NBOX: CK(cudaMemcpy(dst, h->E.nbox, sizeof(int) * n, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_AUX: {
      std::vector<double> tmp((size_t)LLQ_AUX_DIM * n);
      CK(cudaMemcpy(tmp.data(), h->E.aux, sizeof(double) * LLQ_AUX_DIM * n, cudaMemcpyDeviceToHost));
      double* o = (double*)dst;
      for (size_t i = 0; i < n; i++)
        for (int t = 0; t < LLQ_AUX_DIM; t++) o[i * LLQ_AUX_DIM + t] = tmp[(size_t)t * n + i];
      return LLQ_OK;
    }
    case LLQ_F_SAMPLE_PROB:
      if (!h->has_mocap) return fail(LLQ_ESTATE, "no mocap loaded");
      CK(cudaMemcpy(dst, h->d_prob, sizeof(double) * h->n_clips, cudaMemcpyDeviceToHost)); return LLQ_OK;
    case LLQ_F_AVG_REWARD:
      if (!h->has_mocap) return fail(LLQ_ESTATE, "no mocap loaded");
      CK(cudaMemcpy(dst, h->d_avg[h->parity], sizeof(double) * h->n_clips, cudaMemcpyDeviceToHost)); return LLQ_OK;
    default: return fail(LLQ_EINVAL, "unknown field");
  }
}

int llq_set_field(llq_handle h, int field, const void* src) {
  if (!h || !src) return fail(LLQ_EINVAL, "null argument");
  int rc = set_device(h);
  if (rc) return rc;
  const size_t n = (size_t)h->cfg.n_envs;
  CK(cudaStreamSynchronize(h->stream));
  switch (field) {
    case LLQ_F_STATE: {
      const float* s = (const float*)src;
      std::vector<float> st(llq::st::dim * n); std::vector<double> pos(3 * n);
      for (size_t i = 0; i < n; i++) {
        for (int t = 0; t < 3; t++) pos[t * n + i] = (double)s[i * llq::state::dim + llq::state::pos + t];
        for (int t = 0; t < llq::st::dim; t++) st[t * n + i] = s[i * llq::state::dim + llq::state::quat + t];
      }
      CK(cudaMemcpy(h->E.st, st.data(), sizeof(float) * llq::st::dim * n, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(h->E.pos, pos.data(), sizeof(double) * 3 * n, cudaMemcpyHostToDevice));
      return LLQ_OK;
    }
    case LLQ_F_WARMSTART: {
      const float* s = (const float*)src;
      std::vector<float> w(LLQ_MAX_SPHERES * n);
      for (size_t i = 0; i < n; i++) for (int t = 0; t < LLQ_MAX_SPHERES; t++) w[t * n + i] = s[i * LLQ_MAX_SPHERES + t];
      CK(cudaMemcpy(h->E.warm, w.data(), sizeof(float) * LLQ_MAX_SPHERES * n, cudaMemcpyHostToDevice));
      return LLQ_OK;
    }
    case LLQ_F_CLIP: {
      const int* c = (const int*)src;
      for (size_t i = 0; i < n; i++) if (c[i] < 0 || c[i] >= h->n_clips) return fail(LLQ_EINVAL, "clip id out of range");
      CK(cudaMemcpy(h->E.clip, src, sizeof(int) * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    }
    case LLQ_F_TIME: {
      const double* t = (const double*)src;      // the clock indexes the mocap table (ML:65-67): reject what the reference would raise on
      for (size_t i = 0; i < n; i++) if (!(t[i] >= 0.0) || !std::isfinite(t[i])) return fail(LLQ_EINVAL, "env clock must be finite and >= 0");
      CK(cudaMemcpy(h->E.time, src, sizeof(double) * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    }
    case LLQ_F_REWARD_SUM: CK(cudaMemcpy(h->E.reward_sum, src, sizeof(float) * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    case LLQ_F_EPISODE_STEPS: CK(cudaMemcpy(h->E.episode_steps, src, sizeof(int) * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    case LLQ_F_EPISODE_ID: CK(cudaMemcpy(h->E.episode, src, sizeof(long long) * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    case LLQ_F_OB_ID: CK(cudaMemcpy(h->E.ob_id, src, sizeof(int) * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    case LLQ_F_OBS: CK(cudaMemcpy(h->E.obs, src, sizeof(float) * h->obs_dim * n, cudaMemcpyHostToDevice)); return LLQ_OK;
    case LLQ_F_AUX: {
      const double* a = (const double*)src;
      std::vector<double> tmp((size_t)LLQ_AUX_DIM * n);
      for (size_t i = 0; i < n; i++) {
        if (h->cfg.env_kind == LLQ_ENV_EPMC && !(a[i * LLQ_AUX_DIM + 1] >= 1)) return fail(LLQ_EINVAL, "cmd_vary_freq must be positive");
        for (int t = 0; t < LLQ_AUX_DIM; t++) tmp[(size_t)t * n + i] = a[i * LLQ_AUX_DIM + t];
      }
      CK(cudaMemcpy(h->E.aux, tmp.data(), sizeof(double) * LLQ_AUX_DIM * n, cudaMemcpyHostToDevice));
      return LLQ_OK;
    }
    case LLQ_F_SAMPLE_PROB:
      return fail(LLQ_EUNSUPPORTED, "sample probabilities are derived from LLQ_F_AVG_REWARD on the device; set that instead");
    case LLQ_F_AVG_REWARD:
      if (!h->has_mocap) return fail(LLQ_ESTATE, "no mocap loaded");
      CK(cudaMemcpy(h->d_avg[h->parity], src, sizeof(double) * h->n_clips, cudaMemcpyHostToDevice)); return LLQ_OK;
    default: return fail(LLQ_EINVAL, "field is not settable");
  }
}

int llq_get_counters(llq_handle h, int64_t* out, int32_t n) {
  if (!h || !out || n < 0 || n > 8) return fail(LLQ_EINVAL, "bad arguments");
  int rc = set_device(h);
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));
  unsigned long long dc[8];
  CK(cudaMemcpy(dc, h->E.counters, sizeof(dc), cudaMemcpyDeviceToHost));
  int64_t c[8];
  for (int i = 0; i < 8; i++) c[i] = h->counters[i];
  c[1] = (int64_t)dc[1]; c[2] = (int64_t)dc[2]; c[3] = (int64_t)dc[3]; c[5] = (int64_t)dc[5];
  for (int i = 0; i < n; i++) out[i] = c[i];
  return LLQ_OK;
}

int llq_set_option(llq_handle h, const char* name, double value) {
  if (!h || !name) return fail(LLQ_EINVAL, "null argument");
  int rc = set_device(h);
  if (rc) return rc;
  if (!std::strcmp(name, "profile")) {
    h->profile = value != 0;
    if (h->profile && !h->ev[0]) for (int i = 0; i < 3; i++) CK(cudaEventCreate(&h->ev[i]));
    return LLQ_OK;
  }
  if (!std::strcmp(name, "record")) {
    const int v = (int)value;
    if (v < 0 || v > 2) return fail(LLQ_EINVAL, "record must be 0 (off), 1 (same slab row as the observation) or 2 (the row before)");
    h->record = v;
    return LLQ_OK;
  }
  return fail(LLQ_EINVAL, std::string("unknown option ") + name);
}

int llq_get_timing(llq_handle h, double* out, int32_t n) {
  if (!h || !out || n < 2) return fail(LLQ_EINVAL, "bad arguments");
  if (!h->profile || !h->ev_valid) return fail(LLQ_ESTATE, "profiling is off or no step has run");
  int rc = set_device(h);
  if (rc) return rc;
  CK(cudaEventSynchronize(h->ev[2]));
  float a = 0, b = 0;
  CK(cudaEventElapsedTime(&a, h->ev[0], h->ev[1]));
  CK(cudaEventElapsedTime(&b, h->ev[1], h->ev[2]));
  out[0] = a; out[1] = b;
  return LLQ_OK;
}

int llq_host_alloc(void** out, int64_t bytes) {
  if (!out || bytes <= 0) return fail(LLQ_EINVAL, "bad arguments");
  CK(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable));
  return LLQ_OK;
}
int llq_host_free(void* p) {
  if (p) CK(cudaFreeHost(p));
  return LLQ_OK;
}

int llq_sync(llq_handle h) {
  if (!h) return fail(LLQ_EINVAL, "null handle");
  int rc = set_device(h);
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return LLQ_OK;
}

const char* llq_last_error(void) { return g_err.c_str(); }

}  // extern "C"

#ifdef LLQ16_TIMING
// development aid (tools/warp_timing.py): per-warp phase clocks of the last step launch
extern "C" int llq_debug_timing(void* out, int n_warps) {
  return cudaMemcpyFromSymbol(out, llq::g_t16, (size_t)n_warps * 12 * sizeof(unsigned long long)) == cudaSuccess ? 0 : -1;
}
#endif
