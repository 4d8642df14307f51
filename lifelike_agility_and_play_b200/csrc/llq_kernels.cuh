// llq_kernels.cuh -- shared device code of the batched quadruped rollout engine: data layout (model constants, SoA env arrays,
// mocap table), mocap interpolation, Philox streams, ray casting, terrain generation, the observation-row emitter, and the
// reset kernel.  The fused policy-step kernel lives in llq_step16.cuh.
//
// Reset / tail mapping: one environment = 4 adjacent lanes of a warp, one lane per leg (FR, FL, HR, HL); a warp serves 8 environments.
//
// Replaces (reference, relative to src/lifelike/sim_envs/pybullet_envs/):
//   PrimitiveLevelEnv.reset / step tail          primitive_level_env/primitive_level_env.py:150-171, 247-426
//   MotionLib.step/get_states_info(_future)      primitive_level_env/motion_lib.py:48-166
//   PlayGroundEnv reset / perception / rewards   max_game_elements/playground_env.py:196-249, 374-539; bullet_static_entities.py:170-500
//   ChaseTagGameEnv reset / perception / game    max_game/chase_tag_game_env.py:204-304, 472-652
#pragma once
#include "llq_math.cuh"
#include <cuda_pipeline.h>
#include <stdint.h>

namespace llq {

// levels, the ENV argument of the kernel templates: the LLQ_ENV_* kinds, with EPMC split into flat ground (element 0) and the
// corridor arenas of elements 1-3 (static boxes)
constexpr int kPmc = 0, kEpmcFlat = 1, kSepmc = 2, kEpmcCorridor = 3;
constexpr int kObsDim = 207, kObsDimEpmc = 916, kObsDimSepmc = 965, kPropDim = 33, kActDim = 12;
template <int ENV> struct ObsW {
  static constexpr int value = (ENV == kEpmcFlat || ENV == kEpmcCorridor) ? kObsDimEpmc : (ENV == kSepmc ? kObsDimSepmc : kObsDim);
};
constexpr int kMaxBoxes = 36, kMaxCand = 12;   // EPMC corridor: static boxes per env, contact candidates per step
constexpr int kNewObs = 120;
// Staging row: kNewObs floats per robot, written by the tail / reset and read by emit_obs_rows.
//   every level:  prop 33 (joint pos 12 | joint vel 12 | R^T w 3 (24) | R^T v 3 | R[2,:] 3) | action 12 (33)
//   PMC:          future 72 (45)
//   EPMC, SEPMC:  R 9 (45, world <- base inertial, row major) | pos 3 (54), then
//     EPMC:       target direction in the base frame 2 (57) | target speed 1 (59) | |pos| 1 (60) | corridor: yaw 1 (61) | ray masks 3 x 2 (62)
//     SEPMC:      flag xy 2 (57) | yaw 1 (59) | pad 2 | small vectors 52 (62), see sepmc_pair_tail
constexpr int kSlotBase = 24, kSlotFuture = 45, kSlotR = 45, kSlotPos = 54;
constexpr int kSlotTarget = 57, kSlotTargetSpd = 59, kSlotPosLen = 60, kSlotYaw = 61, kSlotMasks = 62;   // EPMC
constexpr int kSlotFlag = 57, kSlotYawSepmc = 59, kSlotVecs = 62;                                          // SEPMC
// rows of E.aux, in the order include/llq.h documents for LLQ_F_AUX; SEPMC gives some rows its own names
namespace aux {
constexpr int counter = 0, cmd_vary_freq = 1, target_x = 2, target_y = 3, target_spd = 4, target_angle = 5, last_pos_diff_len = 6,
              total_spd = 7, max_spd = 8, push_count = 9, push_fx = 10, push_fy = 11, push_fz = 12, foot_friction = 13, push_draws = 14,
              cmd_draws = 15, yaw_accum_deg = 16, init_pos_diff_len = 17;
constexpr int with_flag = 1, flag_x = 2, flag_y = 3, control_spd = 4, oppo_visible = 5, switch_flag = 6, flag_draws = 15, flag_touch = 17;
}  // namespace aux
// rows of the robot state (pybullet base-inertial convention, LR:86-106): LLQ_F_STATE, E.kin and M.init_state use all 37
namespace state {
constexpr int pos = 0, quat = 3, lin = 7, ang = 10, q = 13, qd = 25, dim = 37;
}  // namespace state
// rows of E.st: the same layout without pos, which E.pos keeps in fp64
namespace st {
constexpr int quat = state::quat - 3, lin = state::lin - 3, ang = state::ang - 3, q = state::q - 3, qd = state::qd - 3, dim = state::dim - 3;
}  // namespace st
// record mode: the trajectory columns behind the observation of a slab row, action 12 | reward | done
constexpr int kRecReward = kActDim, kRecDone = kActDim + 1, kRecW = kActDim + 2;

struct DampItem { float m; float c[3]; float Ic[6]; };
struct JointConst {
  float r[3];
  float m; float h[3]; float I[6];
  int nd; DampItem d[2];
  float lower, upper, jdamp; int haslim;
};
struct LegConst { JointConst j[3]; float foot[3]; float foot_r; float pad[4]; };
struct BaseConst { float qI[4]; float m; float h[3]; float I[6]; int nd; DampItem d[3]; };
struct alignas(16) ModelConst {
  BaseConst base; LegConst leg[4];
  float push_R[9]; float push_c[3];   // FR hip link: inertial-frame rotation (link <- inertial) and CoM, for applyExternalForce(LINK_FRAME) (PR:73-77)
  float init_state[state::dim]; float pad_[3]; // EPMC episode start state (LR:115-117, utils/constants.py:103-116)
  // detection proxies for the PMC hurdle plate: wheel (knee) centre in the thigh frame + radius, hip radius, body-box corners (base coords)
  float wheel_off[4][3]; float wheel_r[4]; float hip_r[4]; float corner[8][3];
  float handle[2][4];                  // SEPMC: front / hind handle centre (base coords) + radius (LR:150-156)
};

struct MocapFrame { double x, y, z, pad; float quat[4]; float q[12]; };  // 96 B, 16-byte aligned

struct StepParams {
  int n_envs, substeps, solver_iters;
  float dt, kp, kd, max_tau, gz, mu, erp, jerp, slop, warm, breaking, kl, ka, vmax, max_imp;
  float w_jp, w_jv, w_ee, w_pose, w_vel;   // already normalised to sum 1
  double sim_dt, frame_dt;
  int margin;
  // EPMC (PGE / PR)
  int max_steps, cmd_freq_lo, cmd_freq_hi, push_start_count, push_interval, push_duration, push_enabled;
  float mu_ground, fr_lo, fr_hi, ph_lo, ph_hi, pv_lo, pv_hi, ts_lo, ts_hi;
  // PMC hurdle plates (PLE:173-193)
  int has_ob; float ob_hx, ob_hy, ob_hz;
  // EPMC corridor (BSE)
  int element_id; float ww_lo, ww_hi, wg_lo, wg_hi, hg_lo, hg_hi;
  // knee-wheel ground contact (llq_config.knee_contacts / link_friction)
  int knee; float mu_wheel;
  float aux_r;      // EPMC elements 1-3: radius of the auxiliary edge cylinders (0 = none)
};

struct EnvArrays {      // SoA device arrays, N envs
  double* pos;          // [3][N]
  float* st;            // [34][N]: rows st::
  double* time;         // [N]
  int* clip;            // [N]
  float* reward_sum;    // [N]
  int* episode_steps;   // [N]
  long long* episode;   // [N]
  float* warm;          // [4][N]
  float* obs;           // [N][207] (history carry)
  float* kin;           // [37][N]: rows state::
  float* foot_pos;      // [12][N]
  float* done_reward;   // [N] reward_sum at termination
  unsigned char* done;  // [N]
  float* reward;        // [N]
  unsigned long long* counters;  // [8]
  double* aux;          // [18][N] EPMC bookkeeping (include/llq.h LLQ_F_AUX)
  int* ob_id;           // [N] active hurdle plate
  float* boxes;         // [N][36][6] EPMC corridor: centre xyz, half extents xyz (walls first)
  int* nbox;            // [N]
};

struct MocapDev { const MocapFrame* frames; const int* clip_off; int n_clips; const double* ob_table; const int* ob_off; };

#define FULL 0xffffffffu

LLQ_DI float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }
LLQ_DI float gsum4(float v) {  // sum over the 4 lanes of an env, result on all 4
  v += __shfl_xor_sync(FULL, v, 1);
  v += __shfl_xor_sync(FULL, v, 2);
  return v;
}
LLQ_DI V3 ld3(const float* p) { return V3{p[0], p[1], p[2]}; }
LLQ_DI Sym3 ldsym(const float* p) { return Sym3{p[0], p[1], p[2], p[3], p[4], p[5]}; }

// spatial motion / force vectors (angular, linear) at a link origin, link coordinates
struct SV { V3 a, l; };

// ---------------------------------------------------------------------------------------------------------------
// Mocap interpolation (motion_lib.py:88-166), fp32 except positions/time (fp64)
struct KinBase { double px, py, pz; Q4 q; V3 lin, ang; };

LLQ_DI Q4 ldq(const float* p) { float4 v = *reinterpret_cast<const float4*>(p); return Q4{v.x, v.y, v.z, v.w}; }

LLQ_DI KinBase mocap_base(const MocapFrame* fc, const MocapFrame* fn, double frac, double frame_dt) {
  KinBase k;
  double cx = fc->x, cy = fc->y, cz = fc->z, nx = fn->x, ny = fn->y, nz = fn->z;
  k.px = cx + frac * (nx - cx); k.py = cy + frac * (ny - cy); k.pz = cz + frac * (nz - cz);
  float inv = (float)(1.0 / frame_dt);
  k.lin = V3{(float)(nx - cx) * inv, (float)(ny - cy) * inv, (float)(nz - cz) * inv};
  Q4 qc = qnormalize(ldq(fc->quat)), qn = qnormalize(ldq(fn->quat));
  V3 rv = q_rotvec(qmul(qconj(qc), qn));
  k.q = qmul(qc, rotvec_q((float)frac * rv));
  V3 rw = q_rotvec(qmul(qn, qconj(qc)));
  float angle = norm3(rw);
  float sc = angle / (angle + 1e-8f) * inv;
  k.ang = sc * rw;
  return k;
}

// Foot (link *4) world position for a robot state given in the pybullet base-inertial convention:
// R_bp = world <- B' (URDF body axes), p = base CoM.  q = this leg's joint angles.
LLQ_DI V3 foot_in_base(const LegConst& L, float q1, float q2, float q3) {
  float c1, s1, c2, s2, c3, s3;
  llq_sincosf(q1, &s1, &c1); llq_sincosf(-q2, &s2, &c2); llq_sincosf(-q3, &s3, &c3);
  V3 p = rot<1>(ld3(L.foot), c3, s3) + ld3(L.j[2].r);
  p = rot<1>(p, c2, s2) + ld3(L.j[1].r);
  p = rot<0>(p, c1, s1) + ld3(L.j[0].r);
  return p;
}

// Philox4x32-10
LLQ_DI void philox4x32_10(unsigned (&c)[4], unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    unsigned hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    unsigned hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    unsigned n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

// distance test of a sphere (centre w in world, radius r) against the yawed plate centred at (ox, oy, 0)
LLQ_DI bool plate_hit(V3 w, float r, float cy, float sy, float hx, float hy, float hz, float thr) {
  float bx = cy * w.x + sy * w.y, by = -sy * w.x + cy * w.y;
  float qx = bx - clampf(bx, -hx, hx), qy = by - clampf(by, -hy, hy), qz = w.z - clampf(w.z, -hz, hz);
  return sqrtf(qx * qx + qy * qy + qz * qz) - r < thr;
}

// four uniforms of stream `stream` (1 = EPMC reset, 2 = push randomiser, 3 = joystick command), draw `index` (matches the oracle)
LLQ_DI void stream_uniforms(unsigned long long seed, long long gid, long long episode, unsigned stream, unsigned index, double (&u)[4]) {
  unsigned c[4] = {(unsigned)gid, ((unsigned)((unsigned long long)gid >> 32) & 0x00FFFFFFu) | (stream << 24), (unsigned)episode, index};
  philox4x32_10(c, (unsigned)seed, (unsigned)(seed >> 32));
#pragma unroll
  for (int i = 0; i < 4; i++) u[i] = ((double)c[i] + 0.5) * (1.0 / 4294967296.0);
}
LLQ_DI void epmc_randomize_push(const StepParams& P, unsigned long long seed, long long gid, long long ep, int& push_draws, float (&pf)[3]) {   // PR:89-99
  double u[4];
  stream_uniforms(seed, gid, ep, 2, (unsigned)push_draws++, u);
  double sn, cs;
  sincos(2.0 * 3.14159265358979323846 * u[0], &sn, &cs);
  double h = (double)P.ph_lo + u[1] * ((double)P.ph_hi - (double)P.ph_lo);
  pf[0] = (float)(h * cs); pf[1] = (float)(h * sn); pf[2] = (float)((double)P.pv_lo + u[2] * ((double)P.pv_hi - (double)P.pv_lo));
}

// ---------------------------------------------------------------------------------------------------------------
// Pieces of the step tail and the reset that every level shares.
// Robot state write-back, run on the robot's 4 lanes: this leg's joints and foot (world position), and from lane 0 the base.
LLQ_DI void store_state(const EnvArrays& E, int N, int env, int k, const float (&q)[3], const float (&qd)[3], V3 foot, double px, double py,
                        double pz, Q4 qb, V3 lin, V3 ang) {
  float* sw = E.st;
#pragma unroll
  for (int t = 0; t < 3; t++) { sw[(st::q + 3 * k + t) * N + env] = q[t]; sw[(st::qd + 3 * k + t) * N + env] = qd[t]; }
  E.foot_pos[(3 * k) * N + env] = foot.x; E.foot_pos[(3 * k + 1) * N + env] = foot.y; E.foot_pos[(3 * k + 2) * N + env] = foot.z;
  if (k == 0) {
    E.pos[env] = px; E.pos[N + env] = py; E.pos[2 * N + env] = pz;
    sw[st::quat * N + env] = qb.x; sw[(st::quat + 1) * N + env] = qb.y; sw[(st::quat + 2) * N + env] = qb.z; sw[(st::quat + 3) * N + env] = qb.w;
    sw[st::lin * N + env] = lin.x; sw[(st::lin + 1) * N + env] = lin.y; sw[(st::lin + 2) * N + env] = lin.z;
    sw[st::ang * N + env] = ang.x; sw[(st::ang + 1) * N + env] = ang.y; sw[(st::ang + 2) * N + env] = ang.z;
  }
}
// rotation of the base's inertial frame (pybullet's base orientation) in the URDF body axes: q_inertial = q_body qI
LLQ_DI Q4 base_qI(const ModelConst& M) { return Q4{M.base.qI[0], M.base.qI[1], M.base.qI[2], M.base.qI[3]}; }
// EPMC / SEPMC episode start (LR:115-117): M.init_state with the base yawed by yaw_deg about world z, this leg's joints.  The
// outputs are references, not one returned struct: with the struct, nvcc 12.9 contracts a product of the reset's foot rotation
// into a different FMA, and the reset foot positions change in the last bit.
LLQ_DI Q4 start_pose(const ModelConst& M, int k, double yaw_deg, float (&q)[3], float (&qd)[3], V3& lin, V3& ang) {
  double sn, cs;
  sincos(0.5 * yaw_deg * (3.14159265358979323846 / 180.0), &sn, &cs);
  const float* I0 = M.init_state;
#pragma unroll
  for (int i = 0; i < 3; i++) { q[i] = I0[state::q + 3 * k + i]; qd[i] = I0[state::qd + 3 * k + i]; }
  lin = ld3(I0 + state::lin); ang = ld3(I0 + state::ang);
  const Q4 q0 = Q4{I0[state::quat], I0[state::quat + 1], I0[state::quat + 2], I0[state::quat + 3]};
  return qmul(qnormalize(q0), Q4{0.f, 0.f, (float)sn, (float)cs});
}
// termination on the base orientation (LR:158-179), R = world <- base inertial
LLQ_DI bool fallen(const M3& R) {
  const float left_z = R.a02 * R.a10 - R.a12 * R.a00;
  return left_z > 0.70710678118654752f || left_z < -0.70710678118654752f || R.a22 < 0.5f;
}
// prop base block of a staging row (PLE:247-260): R^T w | R^T v | R[2,:]
LLQ_DI void stage_prop_base(float* snew, const M3& R, V3 ang, V3 lin) {
  const V3 wl = tmul(R, ang), vl = tmul(R, lin);
  float* b = snew + kSlotBase;
  b[0] = wl.x; b[1] = wl.y; b[2] = wl.z; b[3] = vl.x; b[4] = vl.y; b[5] = vl.z;
  b[6] = R.a20; b[7] = R.a21; b[8] = R.a22;
}
// EPMC / SEPMC: the prop base block, then R and pos
LLQ_DI void stage_pose(float* snew, const M3& R, V3 ang, V3 lin, V3 pos) {
  stage_prop_base(snew, R, ang, lin);
  float* r = snew + kSlotR;
  r[0] = R.a00; r[1] = R.a01; r[2] = R.a02; r[3] = R.a10; r[4] = R.a11; r[5] = R.a12; r[6] = R.a20; r[7] = R.a21; r[8] = R.a22;
  snew[kSlotPos] = pos.x; snew[kSlotPos + 1] = pos.y; snew[kSlotPos + 2] = pos.z;
}
// EPMC staging row on lane 0 of the robot: stage_pose, the direction to the target (dx, dy = target - pos) in the base frame, the
// target speed and |pos|
LLQ_DI void stage_epmc(float* snew, const M3& R, V3 ang, V3 lin, double px, double py, double pz, double dx, double dy, float target_spd) {
  stage_pose(snew, R, ang, lin, V3{(float)px, (float)py, (float)pz});
  const V3 d = tmul(R, V3{(float)dx, (float)dy, (float)(0.0 - pz)});
  const float n2 = sqrtf(d.x * d.x + d.y * d.y);
  snew[kSlotTarget] = d.x / n2; snew[kSlotTarget + 1] = d.y / n2; snew[kSlotTargetSpd] = target_spd;
  snew[kSlotPosLen] = (float)sqrt(px * px + py * py + pz * pz);
}

// ---------------------------------------------------------------------------------------------------------------
// SEPMC (ChaseTagGameEnv, max_game/chase_tag_game_env.py = CTG; arena = max_game/bullet_static_entities.py:863-902):
// robots 2p and 2p+1 are the two agents of pair p (adjacent 4-lane groups of one warp).
constexpr float kWallIn = 2.495f;    // inner faces of the four 0.01 m walls centred at +-2.5
// closest hit fraction of the segment o -> o + d against the arena's static boxes (ground slab, 4 walls, flag), or -1
LLQ_DI float ray_box1(V3 o, V3 d, V3 lo, V3 hi, float best) {
  if (o.x > lo.x && o.x < hi.x && o.y > lo.y && o.y < hi.y && o.z > lo.z && o.z < hi.z) return best;   // starts inside: no hit
  float t0 = 0.f, t1 = 1.f;
  bool hit = true, entered = false;
  const float oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z}, l[3] = {lo.x, lo.y, lo.z}, h[3] = {hi.x, hi.y, hi.z};
#pragma unroll
  for (int ax = 0; ax < 3; ax++) {
    if (dd[ax] == 0.f) { if (oo[ax] < l[ax] || oo[ax] > h[ax]) hit = false; continue; }
    const float inv = 1.0f / dd[ax];
    float ta = (l[ax] - oo[ax]) * inv, tb = (h[ax] - oo[ax]) * inv;
    if (ta > tb) { const float t = ta; ta = tb; tb = t; }
    if (ta > t0) { t0 = ta; entered = true; }
    t1 = fminf(t1, tb);
    if (t0 > t1) hit = false;
  }
  if (hit && entered && (best < 0.f || t0 < best)) best = t0;
  return best;
}
// Fast paths of ray_arena for origins inside the arena (|x|, |y| < 2.49): the four walls are then hit on their inner faces, the
// first one crossed is always a valid hit of that face in xy, so only its z range needs checking; same slab arithmetic.
LLQ_DI float ray_arena_inside(V3 o, V3 d, float fx, float fy) {
  float best = -1.f;
  if (d.z < 0.f && o.z > 0.f) {                                    // ground slab top
    const float t = (0.f - o.z) * (1.0f / d.z);
    if (t <= 1.f) best = t;
  }
  float tw = 2.f; 
  if (d.x != 0.f) { const float t = ((d.x > 0.f ? kWallIn : -kWallIn) - o.x) * (1.0f / d.x); tw = t; }
  if (d.y != 0.f) { const float t = ((d.y > 0.f ? kWallIn : -kWallIn) - o.y) * (1.0f / d.y); tw = fminf(tw, t); }
  if (tw <= 1.f) {
    const float z = fmaf(tw, d.z, o.z);
    if (z >= 0.f && z <= 2.f && (best < 0.f || tw < best)) best = tw;
  }
  // the flag is a 0.1 m column: only rays whose line passes within its circumscribed radius (in xy) need the slab test
  const float cx = fx - o.x, cy = fy - o.y, cr = d.x * cy - d.y * cx;
  if (cr * cr > 0.00501f * (d.x * d.x + d.y * d.y)) return best;
  return ray_box1(o, d, V3{fx - 0.05f, fy - 0.05f, 0.f}, V3{fx + 0.05f, fy + 0.05f, 0.5f}, best);
}
LLQ_DI float ray_arena(V3 o, V3 d, float fx, float fy) {
  float b = -1.f;
  b = ray_box1(o, d, V3{-100.f, -100.f, -10.f}, V3{100.f, 100.f, 0.f}, b);
  b = ray_box1(o, d, V3{-2.5f, 2.495f, 0.f}, V3{2.5f, 2.505f, 2.f}, b);
  b = ray_box1(o, d, V3{-2.5f, -2.505f, 0.f}, V3{2.5f, -2.495f, 2.f}, b);
  b = ray_box1(o, d, V3{2.495f, -2.5f, 0.f}, V3{2.505f, 2.5f, 2.f}, b);
  b = ray_box1(o, d, V3{-2.505f, -2.5f, 0.f}, V3{-2.495f, 2.5f, 2.f}, b);
  b = ray_box1(o, d, V3{fx - 0.05f, fy - 0.05f, 0.f}, V3{fx + 0.05f, fy + 0.05f, 0.5f}, b);
  return b;
}
LLQ_DI float flag_dist(V3 c, float fx, float fy) {    // distance of a point to the flag box (CTG:163-190)
  const float qx = c.x - clampf(c.x, fx - 0.05f, fx + 0.05f), qy = c.y - clampf(c.y, fy - 0.05f, fy + 0.05f), qz = c.z - clampf(c.z, 0.f, 0.5f);
  return sqrtf(qx * qx + qy * qy + qz * qz);
}
// points of this lane's leg in base coordinates (B' axes about the base reference point)
LLQ_DI void leg_points(const ModelConst& M, const LegConst& L, int k, const float (&q)[3], V3& hip, V3& wheel, V3& foot) {
  float c1, s1, c2, s2, c3, s3;
  llq_sincosf(q[0], &s1, &c1); llq_sincosf(-q[1], &s2, &c2); llq_sincosf(-q[2], &s3, &c3);
  hip = ld3(L.j[0].r);
  const V3 p2 = hip + rot<0>(ld3(L.j[1].r), c1, s1);
  wheel = p2 + rot<0>(rot<1>(ld3(M.wheel_off[k]), c2, s2), c1, s1);
  V3 f = rot<1>(ld3(L.foot), c3, s3) + ld3(L.j[2].r);
  f = rot<1>(f, c2, s2) + ld3(L.j[1].r);
  foot = rot<0>(f, c1, s1) + hip;
}

// small vectors of the SEPMC staging row (kSlotVecs): percept_vec 5, oppo_info 15, oppo_info_cheat 15, flag_info 7, flag_info_cheat 7,
// with_flag 2, control_spd 1
struct PairState { int with_flag, flag_draws, visible, sw; double flag_x, flag_y; };

// End-of-step pair logic shared by the step and the reset kernels (CTG:495-596, 472-493): visibility, flag switch, the small
// observation vectors.  Every lane of both robots runs it (the partner robot is 4 lanes away); `snew` is the robot's staging row,
// `spart` the partner's.
LLQ_DI void sepmc_pair_tail(const ModelConst& M, const LegConst& L, int k, int robot, float* snew, const float* spart, double px, double py,
                            double pz, Q4 qp, Q4 qb, V3 vw, V3 ww, const float (&q)[3], bool touch_own, float fix_spd, unsigned long long seed,
                            long long pair_gid, long long epi, PairState& S) {
  const M3 Rp = qmat(qp);
  const V3 pos = V3{(float)px, (float)py, (float)pz};
  // own convex points (LR:150-156) in world coordinates -> staging row, read by the partner
  {
    V3 hip, wheel, foot;
    leg_points(M, L, k, q, hip, wheel, foot);
    const V3 fw = pos + mul(Rp, foot), ww_ = pos + mul(Rp, wheel);
    snew[3 * k] = fw.x; snew[3 * k + 1] = fw.y; snew[3 * k + 2] = fw.z;
    snew[12 + 3 * k] = ww_.x; snew[13 + 3 * k] = ww_.y; snew[14 + 3 * k] = ww_.z;
    if (k < 2) {
      const V3 hw = pos + mul(Rp, V3{M.handle[k][0], M.handle[k][1], M.handle[k][2]});
      snew[24 + 3 * k] = hw.x; snew[25 + 3 * k] = hw.y; snew[26 + 3 * k] = hw.z;
    }
  }
  __syncwarp();
  // partner's root state
  const double ox = __shfl_xor_sync(FULL, px, 4), oy = __shfl_xor_sync(FULL, py, 4), oz = __shfl_xor_sync(FULL, pz, 4);
  const Q4 oq = Q4{__shfl_xor_sync(FULL, qb.x, 4), __shfl_xor_sync(FULL, qb.y, 4), __shfl_xor_sync(FULL, qb.z, 4), __shfl_xor_sync(FULL, qb.w, 4)};
  const V3 ov = V3{__shfl_xor_sync(FULL, vw.x, 4), __shfl_xor_sync(FULL, vw.y, 4), __shfl_xor_sync(FULL, vw.z, 4)};
  const V3 oww = V3{__shfl_xor_sync(FULL, ww.x, 4), __shfl_xor_sync(FULL, ww.y, 4), __shfl_xor_sync(FULL, ww.z, 4)};
  const bool touch_other = __shfl_xor_sync(FULL, touch_own ? 1 : 0, 4) != 0;
  const V3 opos = V3{(float)ox, (float)oy, (float)oz};
  const float fx = (float)S.flag_x, fy = (float)S.flag_y;
  // visibility (CTG:472-493): the root segment is cast from robot 0 to robot 1 for both agents
  const V3 ra = robot == 0 ? pos : opos, rb = robot == 0 ? opos : pos;
  bool vis = ray_arena(ra, rb - ra, fx, fy) < 0.f;
  {
    const V3 head = V3{snew[24], snew[25], snew[26]};
    const V3 tf = V3{spart[3 * k], spart[3 * k + 1], spart[3 * k + 2]}, tw = V3{spart[12 + 3 * k], spart[13 + 3 * k], spart[14 + 3 * k]};
    bool any = ray_arena(head, tf - head, fx, fy) < 0.f || ray_arena(head, tw - head, fx, fy) < 0.f;
    if (k < 2) {
      const V3 th = V3{spart[24 + 3 * k], spart[25 + 3 * k], spart[26 + 3 * k]};
      any = any || ray_arena(head, th - head, fx, fy) < 0.f;
    }
    int a = any ? 1 : 0;
    a |= __shfl_xor_sync(FULL, a, 1);
    a |= __shfl_xor_sync(FULL, a, 2);
    vis = vis || a != 0;
  }
  const Q4 q1 = qnormalize(qb);
  const M3 Rq = qmat(q1);
  {
    // cos of the bearing of the opponent against visible_angle = pi; in fp64 so that |cos| <= 1 holds unless fp64 itself rounds over
    const double c = (double)Rq.a00, s_ = (double)Rq.a10, n = sqrt(c * c + s_ * s_);
    const double dx = ox - px, dy = oy - py;
    const double cv = ((c / n) * dx + (s_ / n) * dy) / sqrt(dx * dx + dy * dy);
    vis = vis && cv >= -1.0;
  }
  __syncwarp();   // convex points consumed; the row is free for the observation staging
  S.visible = vis ? 1 : 0;
  // flag switch (CTG:573-581): the robot without the flag touches it
  const int wf_old = S.with_flag;
  const double ffx = S.flag_x, ffy = S.flag_y;
  S.sw = 0;
  if ((wf_old && touch_other) || (!wf_old && touch_own)) {
    S.with_flag = 1 - wf_old;
    S.sw = 1;
    double u[4];
    stream_uniforms(seed, pair_gid, epi, 4, (unsigned)S.flag_draws, u);
    S.flag_draws += 1;
    S.flag_x = -2.0 + 4.0 * u[0]; S.flag_y = -2.0 + 4.0 * u[1];
  }
  if (k == 0) {
    stage_pose(snew, Rq, ww, vw, pos);
    snew[kSlotFlag] = (float)ffx; snew[kSlotFlag + 1] = (float)ffy;     // the flag where it stood during this step
    const float yaw = atan2f(Rq.a10, Rq.a00);
    snew[kSlotYawSepmc] = yaw;
    float sy, cy;
    llq_sincosf(yaw, &sy, &cy);
    float* v = snew + kSlotVecs;
    v[0] = pos.x; v[1] = pos.y; v[2] = pos.z; v[3] = cy; v[4] = sy;                          // percept_vec
    const M3 Ro = qmat(qnormalize(oq));
    const float yawo = atan2f(Ro.a10, Ro.a00);
    float sd, cd;
    llq_sincosf(yawo - yaw, &sd, &cd);
    const V3 dl = tmul(Rq, V3{(float)(ox - px), (float)(oy - py), (float)(oz - pz)}), ovl = tmul(Rq, ov), owl = tmul(Rq, oww);
    const float oppo[15] = {vis ? 1.f : 0.f, opos.x, opos.y, opos.z, dl.x, dl.y, dl.z, cd, sd, ovl.x, ovl.y, ovl.z, owl.x, owl.y, owl.z};
#pragma unroll
    for (int t = 0; t < 15; t++) { v[5 + t] = vis ? oppo[t] : 0.f; v[20 + t] = oppo[t]; }
    const V3 fl = tmul(Rq, V3{(float)(ffx - px), (float)(ffy - py), (float)(0.25 - pz)});
    const float fi[7] = {1.f, (float)ffx, (float)ffy, 0.25f, fl.x, fl.y, fl.z};
#pragma unroll
    for (int t = 0; t < 7; t++) { v[35 + t] = fi[t]; v[42 + t] = fi[t]; }
    v[49] = (float)S.with_flag; v[50] = (float)(1 - S.with_flag);                              // CTG:584, after a possible switch
    v[51] = fix_spd;
  }
}


// ---------------------------------------------------------------------------------------------------------------
// EPMC corridor (elements 1-3; BSE = max_game_elements/bullet_static_entities.py).
// 64-bit mask of the env's boxes whose xy footprint comes within `margin` of (px, py) (zsel: whose z range contains pz);
// the 4 lanes of an env scan interleaved quarters and combine.
LLQ_DI unsigned long long box_mask(const float* boxes, int nb, int k, float px, float py, float pz, float margin, bool zsel) {
  unsigned long long m = 0ull;
  for (int j = k; j < nb; j += 4) {
    const float* b = boxes + 6 * j;
    const bool hit = zsel ? fabsf(b[2] - pz) <= b[5] : (fabsf(b[0] - px) <= b[3] + margin && fabsf(b[1] - py) <= b[4] + margin);
    if (hit) m |= 1ull << j;
  }
  unsigned lo = (unsigned)m, hi = (unsigned)(m >> 32);
  lo |= __shfl_xor_sync(FULL, lo, 1); hi |= __shfl_xor_sync(FULL, hi, 1);
  lo |= __shfl_xor_sync(FULL, lo, 2); hi |= __shfl_xor_sync(FULL, hi, 2);
  return ((unsigned long long)hi << 32) | lo;
}
// closest hit fraction against the ground slab and the boxes selected by `mask`.  A box whose bounds lie clear (by more than 0.1 mm:
// grazing cases stay with the slab test) of the segment's own bounds cannot be hit and is skipped before the slab test.
LLQ_DI float ray_boxlist(V3 o, V3 d, const float* boxes, unsigned long long mask) {
  float best = ray_box1(o, d, V3{-100.f, -100.f, -10.f}, V3{100.f, 100.f, 0.f}, -1.f);
  const float ex = o.x + d.x, ey = o.y + d.y, ez = o.z + d.z;
  const float x0 = fminf(o.x, ex) - 1e-4f, x1 = fmaxf(o.x, ex) + 1e-4f, y0 = fminf(o.y, ey) - 1e-4f, y1 = fmaxf(o.y, ey) + 1e-4f;
  const float z0 = fminf(o.z, ez) - 1e-4f, z1 = fmaxf(o.z, ez) + 1e-4f;
  while (mask) {
    const int j = __ffsll((long long)mask) - 1;
    mask &= mask - 1;
    const float* b = boxes + 6 * j;
    const V3 lo = V3{b[0] - b[3], b[1] - b[4], b[2] - b[5]}, hi = V3{b[0] + b[3], b[1] + b[4], b[2] + b[5]};
    if (lo.x > x1 || hi.x < x0 || lo.y > y1 || hi.y < y0 || lo.z > z1 || hi.z < z0) continue;
    best = ray_box1(o, d, lo, hi, best);
  }
  return best;
}
// a vertical ray from z = 10 down to z = -10 at (x, y): the z of what it hits first = the highest top among the ground slab and the
// selected boxes whose footprint holds (x, y) (same inclusive bounds as the slab test); < 0: nothing (off the slab)
LLQ_DI float down_ray_top(float x, float y, const float* boxes, unsigned long long mask) {
  float top = (x < -100.f || x > 100.f || y < -100.f || y > 100.f) ? -1.f : 0.f;
  while (mask) {
    const int j = __ffsll((long long)mask) - 1;
    mask &= mask - 1;
    const float* b = boxes + 6 * j;
    const bool out = x < b[0] - b[3] || x > b[0] + b[3] || y < b[1] - b[4] || y > b[1] + b[4];
    if (!out) top = fmaxf(top, b[2] + b[5]);
  }
  return top;
}
struct TerrainRng {
  unsigned long long seed; long long gid, ep; int k; double u[4];
  LLQ_DI double next() {
    if ((k & 3) == 0) stream_uniforms(seed, gid, ep, 5, (unsigned)(k >> 2), u);
    const double v = (k & 3) == 0 ? u[0] : ((k & 3) == 1 ? u[1] : ((k & 3) == 2 ? u[2] : u[3]));
    k++;
    return v;
  }
  LLQ_DI double uniform(double lo, double hi) { return lo + next() * (hi - lo); }
  LLQ_DI int randint(int lo, int hi) { return lo + (int)floor(next() * (double)(hi - lo)); }
};
LLQ_DI void put_box(float* boxes, int& nb, bool wr, double cx, double cy, double cz, double lx, double ly, double lz) {
  if (nb < kMaxBoxes && wr) {
    float* b = boxes + 6 * nb;
    b[0] = (float)cx; b[1] = (float)cy; b[2] = (float)cz; b[3] = (float)(lx / 2); b[4] = (float)(ly / 2); b[5] = (float)(lz / 2);
  }
  if (nb < kMaxBoxes) nb++;
}
// reset(): _generate_random_width_walls + _create_hurdles / _create_holes / _create_cubes(easy) (BSE:170-263, 308-500); returns the
// number of boxes, writes them when `wr`, and the target x (target y = 0)
LLQ_DI int generate_corridor(const StepParams& P, unsigned long long seed, long long gid, long long ep, float* boxes, bool wr, double& tgx) {
  TerrainRng R{seed, gid, ep, 0, {0.0, 0.0, 0.0, 0.0}};
  int nb = 0;
  const double width = R.uniform((double)P.ww_lo, (double)P.ww_hi), gap = R.uniform((double)P.wg_lo, (double)P.wg_hi);
  put_box(boxes, nb, wr, 5.0, gap / 2.0 + width / 2.0, 1.0, 200.0, width, 2.0);
  put_box(boxes, nb, wr, 5.0, -(gap / 2.0 + width / 2.0), 1.0, 200.0, width, 2.0);
  double cur = 0.0;
  tgx = 8.0;
  if (P.element_id == 1 || P.element_id == 2) {
    const int n = R.randint(1, 10);
    for (int pass = 0; pass < 2; pass++) {
      for (int i = 0; i < n; i++) {
        if (P.element_id == 1) {
          const double h = R.uniform(0.05, 0.15), d = R.uniform(1.0, 3.0);
          put_box(boxes, nb, wr, cur + d / 2, 0.0, h / 2, 0.1, gap, h);
          cur += d + 0.1;
        } else {
          const double d = R.uniform(1.0, 3.0), g = R.uniform((double)P.hg_lo, (double)P.hg_hi);
          put_box(boxes, nb, wr, cur + d / 2, 0.0, 0.3 / 2 + g, 0.1, gap, 0.3);
          cur += d + 0.1;
        }
      }
      if (pass == 0) tgx = cur + R.uniform(-1.0, 1.0);
    }
  } else {
    const int ns = R.randint(1, 5);
    for (int pass = 0; pass < 2; pass++) {
      for (int i = 0; i < ns; i++) {
        cur += R.uniform(0.0, 1.0);
        put_box(boxes, nb, wr, 1.75 + cur, 0.0, 0.25 / 2, 0.5, gap, 0.25);
        put_box(boxes, nb, wr, 1.0 + cur, 0.0, 0.1 / 2, 0.5, gap, 0.1);
        cur += 1.75 + 0.25;
        put_box(boxes, nb, wr, cur + 0.5, 0.0, 0.25 / 2, 0.5, gap, 0.25);
        put_box(boxes, nb, wr, cur + 1.25, 0.0, 0.1 / 2, 0.5, gap, 0.1);
        cur += 3.0;
      }
      if (pass == 0) tgx = cur + R.uniform(-3.0, 3.0);
    }
  }
  return nb;
}
// stage the perception context of an EPMC-corridor row: yaw and the three candidate masks (as raw bits)
LLQ_DI void stage_corridor_masks(float* snew, const float* boxes, int nb, int k, float px, float py, float pz, float yaw) {
  const unsigned long long m2 = box_mask(boxes, nb, k, px, py, pz, 1.36f, false);   // 2.4 x 1.2 footprint, any yaw
  const unsigned long long mf = box_mask(boxes, nb, k, px, py, pz, 3.35f, false);   // 3 m rays starting up to 0.27 m off the base
  const unsigned long long m1 = box_mask(boxes, nb, k, px, py, pz, 0.f, true);      // horizontal rays at the base height
  if (k == 0) {
    float* m = snew + kSlotMasks;
    snew[kSlotYaw] = yaw;
    m[0] = __uint_as_float((unsigned)m2); m[1] = __uint_as_float((unsigned)(m2 >> 32));
    m[2] = __uint_as_float((unsigned)mf); m[3] = __uint_as_float((unsigned)(mf >> 32));
    m[4] = __uint_as_float((unsigned)m1); m[5] = __uint_as_float((unsigned)(m1 >> 32));
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Shared tail: given the dynamic robot state (pybullet convention) and the mocap cursor, build the new prop / future
// into the staging row `snew` (120 floats per env) and return the pieces the reward needs.
struct ObsCtx {
  KinBase kb;          // kinematic (mocap) base
  float kq[3], kqd[3]; // kinematic joints of this lane's leg
};

LLQ_DI ObsCtx build_obs_new(const MocapDev& mc, const StepParams& P, const ModelConst& M, int lane4, int clip, int frame_id,
                            double frac, double px, double py, double pz, Q4 qb, V3 lin, V3 ang, const float (&q)[3],
                            const float (&qd)[3], float* snew) {
  ObsCtx o;
  const MocapFrame* f0 = mc.frames + mc.clip_off[clip] + frame_id;
  o.kb = mocap_base(f0, f0 + 1, frac, P.frame_dt);
  float inv = (float)(1.0 / P.frame_dt), fr = (float)frac;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    float c = f0->q[3 * lane4 + i], n = f0[1].q[3 * lane4 + i];
    o.kq[i] = fmaf(fr, n - c, c);
    o.kqd[i] = (n - c) * inv;
  }
  qb = qnormalize(qb);
  M3 Rb = qmat(qb);
  // prop (PLE:247-260): joint_pos | joint_vel | R^T w | R^T v | R[2,:]
#pragma unroll
  for (int i = 0; i < 3; i++) { snew[3 * lane4 + i] = q[i]; snew[12 + 3 * lane4 + i] = qd[i]; }
  if (lane4 == 0) stage_prop_base(snew, Rb, ang, lin);
  // future target `lane4` (ML:75-86, PLE:299-317)
  {
    const double tf = lane4 == 0 ? 1. / 30. : (lane4 == 1 ? 1. / 15. : (lane4 == 2 ? 1. / 3. : 1.));
    double t = P.frame_dt * frac + tf;
    int fid = (int)floor(t / P.frame_dt);
    double ffrac = t / P.frame_dt - fid;
    const MocapFrame* g0 = f0 + fid;
    KinBase kf = mocap_base(g0, g0 + 1, ffrac, P.frame_dt);
    V3 dp = tmul(Rb, V3{(float)(kf.px - px), (float)(kf.py - py), (float)(kf.pz - pz)});
    V3 rv = q_rotvec(qnormalize(qmul(qconj(qb), qnormalize(kf.q))));
    float angle = norm3(rv);
    float sc = angle / (angle + 1e-8f);
    float* o18 = snew + kSlotFuture + 18 * lane4;
    o18[0] = dp.x; o18[1] = dp.y; o18[2] = dp.z;
    o18[3] = sc * rv.x; o18[4] = sc * rv.y; o18[5] = sc * rv.z;
    float ff = (float)ffrac;
#pragma unroll
    for (int j = 0; j < 12; j++) { float c = g0->q[j], n = g0[1].q[j]; o18[6 + j] = fmaf(ff, n - c, c); }
  }
  return o;
}

// Cooperative, coalesced emission of the 8 observation rows owned by this warp.
// mode 0 (step):  prop = [old[33:99], new] ; prop_a = [old[12:36], act] ; future = new
// mode 1 (reset): prop = [new, new, new]  ; prop_a = 0                 ; future = new      (PLE:282-290)
// `do_row` (bit e of a warp-uniform mask) selects which of the 8 rows are written.  EPMC / SEPMC: the perception rays are cast
// while the row is written.
constexpr int kHist = 90;   // per-env history carry: prop[33:99] (66) | prop_a[12:36] (24)

// Perception ray geometry from the R and pos slots of an EPMC / SEPMC staging row (PGE:409-447).
// down ray t of percept_2d, over the 25 x 13 grid of 2.4 x 1.2 m in the base frame: its world xy
LLQ_DI void down_ray_xy(const float* sn, int t, float& x, float& y) {
  const float* R = sn + kSlotR;
  const int a = t / 13, b = t - a * 13;
  const float gx = a == 24 ? 1.2f : -1.2f + (float)a * (2.4f / 24.0f), gy = b == 12 ? 0.6f : -0.6f + (float)b * (1.2f / 12.0f);
  x = fmaf(R[0], gx, fmaf(R[1], gy, sn[kSlotPos])); y = fmaf(R[3], gx, fmaf(R[4], gy, sn[kSlotPos + 1]));
}
// front ray t of percept_front: origins on the 25 x 13 grid over base y in [-0.25, 0.25], z in [-0.3, 0.1]; 3 m along base +x
LLQ_DI void front_ray(const float* sn, int t, V3& from, V3& d) {
  const float* R = sn + kSlotR;
  const int a = t / 13, b = t - a * 13;
  const float y = a == 24 ? 0.25f : -0.25f + (float)a * (0.5f / 24.0f), z = b == 12 ? 0.1f : -0.3f + (float)b * (0.4f / 12.0f);
  from = V3{fmaf(R[1], y, fmaf(R[2], z, sn[kSlotPos])), fmaf(R[4], y, fmaf(R[5], z, sn[kSlotPos + 1])),
            fmaf(R[7], y, fmaf(R[8], z, sn[kSlotPos + 2]))};
  d = V3{3.f * R[0], 3.f * R[3], 3.f * R[6]};
}
template <int ENV, int EPW = 8>   // EPW = envs per warp (8 with 4 lanes per env, 2 with 16)
LLQ_DI void emit_obs_rows(float* obs, float* obs2, long long obs2_ld, const float* snew_warp, const float* hist_warp, int env0, int n_envs,
                          int mode, unsigned row_mask, const float* boxes_all = nullptr) {
  constexpr int OW = ObsW<ENV>::value;
  const int lane = threadIdx.x & 31;
#pragma unroll 4
  for (int base = 0; base < EPW * OW; base += 32) {
    int idx = base + lane;
    int e = idx / OW, j = idx - e * OW;
    bool ok = idx < EPW * OW && (env0 + e) < n_envs && ((row_mask >> e) & 1u);
    float v = 0.f;
    if (ok) {
      const float* sn = snew_warp + e * kNewObs;
      const float* hs = hist_warp + e * kHist;
      if (j < 99) {
        if (mode == 1) v = sn[j % kPropDim];
        else v = j < 66 ? hs[j] : sn[j - 66];
      } else if (j < 135) {
        int a = j - 99;
        if (mode == 1) v = 0.f;
        else v = a < 24 ? hs[66 + a] : sn[kPropDim + a - 24];
      } else if (ENV == kPmc) {
        v = sn[kSlotFuture + (j - 135)];
      } else if (ENV == kEpmcCorridor) {
        // EPMC corridor perception against the ground slab and the env's candidate boxes (PGE:374-447)
        const V3 pos = ld3(sn + kSlotPos);
        const float* bxs = boxes_all + (size_t)(env0 + e) * (6 * kMaxBoxes);
        const float* ms = sn + kSlotMasks;
        if (j < 460) {
          const unsigned long long m = ((unsigned long long)__float_as_uint(ms[1]) << 32) | __float_as_uint(ms[0]);
          float x, y;
          down_ray_xy(sn, j - 135, x, y);
          v = fmaxf(down_ray_top(x, y, bxs, m), 0.f);          // hit z of the down ray (0 when it misses everything)
        } else if (j < 588) {
          const unsigned long long m = ((unsigned long long)__float_as_uint(ms[5]) << 32) | __float_as_uint(ms[4]);
          const float ang = sn[kSlotYaw] + 6.283185307179586f * (float)(j - 460) * (1.0f / 128.0f);
          float sa, ca;
          llq_sincosf(ang, &sa, &ca);
          const float f = ray_boxlist(pos, V3{20.f * ca, 20.f * sa, 0.f}, bxs, m);
          v = f < 0.f ? sn[kSlotPosLen] : f * 20.f * sqrtf(ca * ca + sa * sa);
        } else if (j < 913) {
          const unsigned long long m = ((unsigned long long)__float_as_uint(ms[3]) << 32) | __float_as_uint(ms[2]);
          V3 from, d;
          front_ray(sn, j - 588, from, d);
          const float f = ray_boxlist(from, d, bxs, m);
          v = (f < 0.f ? 1.f : f) * norm3(d);
        } else {
          v = sn[kSlotTarget + (j - 913)];
        }
      } else if (ENV == kSepmc) {
        // SEPMC perception against ground slab, walls and flag (CTG:598-638, PGE:22-54)
        const V3 pos = ld3(sn + kSlotPos);
        const float fx = sn[kSlotFlag], fy = sn[kSlotFlag + 1];
        if (j < 460) {                             // percept_2d: down rays over the 25 x 13 grid in the full base frame, value = hit z
          float x, y;
          down_ray_xy(sn, j - 135, x, y);
          // a vertical ray sees the highest top among the boxes whose footprint holds (x, y): flag 0.5, walls 2, ground 0
          const bool in_x = fabsf(x) <= 2.5f, in_y = fabsf(y) <= 2.5f;
          const bool wall = (in_x && fabsf(fabsf(y) - 2.5f) <= 0.005f) || (in_y && fabsf(fabsf(x) - 2.5f) <= 0.005f);
          const bool flag = fabsf(x - fx) <= 0.05f && fabsf(y - fy) <= 0.05f;
          v = wall ? 2.0f : (flag ? 0.5f : 0.0f);
          if (!(fabsf(x) < 99.f && fabsf(y) < 99.f)) {                    // off the slab: the general test decides
            const float f = ray_arena(V3{x, y, 10.f}, V3{0.f, 0.f, -20.f}, fx, fy);
            v = f < 0.f ? 0.f : fmaf(f, -20.f, 10.f);
          }
        } else if (j < 588) {                      // percept_1d: 128 horizontal rays of 20 m; a miss reports |ray_from|
          const float ang = sn[kSlotYawSepmc] + 6.283185307179586f * (float)(j - 460) * (1.0f / 128.0f);
          float sa, ca;
          llq_sincosf(ang, &sa, &ca);
          const V3 d = V3{20.f * ca, 20.f * sa, 0.f};
          const bool inside = fabsf(pos.x) < 2.49f && fabsf(pos.y) < 2.49f;
          const float f = inside ? ray_arena_inside(pos, d, fx, fy) : ray_arena(pos, d, fx, fy);
          v = f < 0.f ? norm3(pos) : f * 20.f * sqrtf(ca * ca + sa * sa);
        } else if (j < 913) {                      // percept_front: 25 x 13 rays of 3 m along body +x; a miss reports 3
          V3 from, d;
          front_ray(sn, j - 588, from, d);
          const bool inside = fabsf(from.x) < 2.49f && fabsf(from.y) < 2.49f && from.z > 0.f;
          const float f = inside ? ray_arena_inside(from, d, fx, fy) : ray_arena(from, d, fx, fy);
          v = (f < 0.f ? 1.f : f) * norm3(d);
        } else {
          v = sn[kSlotVecs + (j - 913)];
        }
      } else if (j < 460) {
        v = 0.f;                                   // percep_2d: every down-ray hits the slab top, hit z = 0 (PGE:431-447)
      } else if (j < 588) {
        v = sn[kSlotPosLen];                       // percep_1d: horizontal rays miss => |ray_from| (PGE:49-53,388-394)
      } else if (j < 913) {                        // percep_front (PGE:409-429) against the ground slab
        const float* R = sn + kSlotR;
        int t = j - 588, i = t / 13, jj = t - i * 13;
        float y = i == 24 ? 0.25f : -0.25f + (float)i * (0.5f / 24.0f);
        float z = jj == 12 ? 0.1f : -0.3f + (float)jj * (0.4f / 12.0f);
        float fz = fmaf(R[7], y, fmaf(R[8], z, sn[kSlotPos + 2]));   // from.z = R[2,1] y + R[2,2] z + pos.z
        float dz = 3.0f * R[6];                                       // (to - from).z = 3 R[2,0]
        float len = 3.0f * sqrtf(R[0] * R[0] + R[3] * R[3] + R[6] * R[6]);
        float tz = fz + dz;
        v = (fz > 0.f && tz < 0.f) ? len * (fz / (fz - tz)) : len;
      } else {
        v = sn[kSlotTarget + (j - 913)];
      }
      obs[(size_t)(env0 + e) * OW + j] = v;
      if (obs2) obs2[(size_t)(env0 + e) * obs2_ld + j] = v;
    }
  }
}

// Asynchronous (cp.async) prefetch issued at kernel start; consumed after the ten sub-steps, so DRAM latency is hidden.
template <int ENV, int EPW = 8>
LLQ_DI void prefetch_history(const float* obs, float* hist_warp, int env0, int n_envs) {
  constexpr int OW = ObsW<ENV>::value;
  const int lane = threadIdx.x & 31;
  for (int idx = lane; idx < EPW * kHist; idx += 32) {
    int e = idx / kHist, t = idx - e * kHist;
    int env = env0 + e < n_envs ? env0 + e : n_envs - 1;
    int j = t < 66 ? 33 + t : 99 + 12 + (t - 66);
    __pipeline_memcpy_async(hist_warp + idx, obs + (size_t)env * OW + j, 4);
  }
}
LLQ_DI void prefetch_model(const ModelConst* gmodel, ModelConst* smodel, int nthreads) {
  static_assert(sizeof(ModelConst) % 16 == 0, "ModelConst must be a multiple of 16 bytes");
  const float4* src = reinterpret_cast<const float4*>(gmodel);
  float4* dst = reinterpret_cast<float4*>(smodel);
  for (int i = threadIdx.x; i < (int)(sizeof(ModelConst) / 16); i += nthreads) __pipeline_memcpy_async(dst + i, src + i, 16);
}

// ---------------------------------------------------------------------------------------------------------------
// Reset kernel (PLE:150-171, ML:48-63): also owns the prioritized-sampling table update (PLE:235-240).
// mode 0: reset envs with done[i] != 0 (auto-reset after a step), sampling clip/phase
// mode 1: reset envs with mask[i] != 0 (mask == null: all), sampling
// mode 2: like mode 1 but clip/time given
// mode 3: no env is reset (table update only; auto_reset off)
struct ResetParams {
  int mode; const unsigned char* mask; const int* clip_in; const double* time_in;
  unsigned long long seed; long long gid0;
  int* winner_cur; int* winner_next;          // [n_clips]
  const double* avg_old; double* avg_new;     // [n_clips]
  double* prob;                               // [n_clips]  (written by block 0)
  const double* max_steps;                    // [n_clips]
  double factor;
  int update_table;                           // 1 after a step
};

template <int BLOCK, int ENV>
__global__ void __launch_bounds__(BLOCK) pmc_reset_kernel(EnvArrays E, MocapDev mc, StepParams P, const ModelConst* __restrict__ gmodel,
                                                          ResetParams RP, float* obs2, long long obs2_ld) {
  extern __shared__ double s_cdf[];            // [n_clips]
  __shared__ __align__(16) ModelConst M;
  __shared__ __align__(16) float s_new[BLOCK / 4][kNewObs];
  prefetch_model(gmodel, &M, BLOCK);
  __pipeline_commit();
  const int C = mc.n_clips;
  // ---- prioritized sampling table: every block recomputes it identically; block 0 publishes it
  for (int c = threadIdx.x; c < C; c += BLOCK) {
    double avg = RP.avg_old[c];
    if (RP.update_table) {
      int w = RP.winner_cur[c];
      if (w >= 0) avg = (double)E.done_reward[w] / RP.max_steps[c];
    }
    s_cdf[c] = avg;
  }
  __syncthreads();
  if (RP.update_table && blockIdx.x == 0)
    for (int c = threadIdx.x; c < C; c += BLOCK) { RP.avg_new[c] = s_cdf[c]; RP.winner_next[c] = -1; }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += BLOCK) s_cdf[c] = pow(1.0 - s_cdf[c], RP.factor);
  __syncthreads();
  // p = w / sum(w), cdf = cumsum(p) / cumsum(p)[-1] exactly as np.random.choice builds them: the two sums run sequentially on one
  // thread (their order fixes the last bits), the 2 C fp64 divisions -- 3/4 of this section's latency when thread 0 did them one
  // after the other -- run one per thread
  __shared__ double s_tot;
  if (threadIdx.x == 0) {
    double tot = 0;
    for (int c = 0; c < C; c++) tot += s_cdf[c];
    s_tot = tot;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += BLOCK) {
    const double pc = s_cdf[c] / s_tot;
    s_cdf[c] = pc;
    if (blockIdx.x == 0) RP.prob[c] = pc;
  }
  __syncthreads();
  if (threadIdx.x == 0 && C > 0) {
    double acc = 0;
    for (int c = 0; c < C; c++) { acc += s_cdf[c]; s_cdf[c] = acc; }
    s_tot = s_cdf[C - 1];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += BLOCK) s_cdf[c] = s_cdf[c] / s_tot;
  __syncthreads();

  __pipeline_wait_prior(0);
  __syncthreads();
  const int N = P.n_envs;
  const int gtid = blockIdx.x * BLOCK + threadIdx.x;
  const int env_raw = gtid >> 2;
  const int env = env_raw < N ? env_raw : N - 1;
  const bool valid = env_raw < N;
  const int k = threadIdx.x & 3;
  bool doit = valid;
  if (RP.mode == 3) doit = false;
  else if (RP.mode == 0) doit = doit && E.done[env] != 0;
  else if (RP.mask) doit = doit && (RP.mask[env] != 0 || (ENV == kSepmc && RP.mask[env ^ 1] != 0));   // SEPMC: a pair resets as a whole
  const unsigned wm = __ballot_sync(FULL, doit);
  if (wm == 0) return;                                   // warp-uniform: nothing to reset in these 8 envs
  const LegConst& L = M.leg[k];

  if (ENV == kSepmc) {
    // ---------------- SEPMC reset (CTG:261-304, 204-230); draws keyed by the pair: stream 1 = [fix_spd, with_flag, friction, x0 |
    // y0, x1, y1, yaw0 | yaw1, flag x, flag y]
    const int robot = env & 1;
    const long long ep = E.episode[env];
    const long long gid = RP.gid0 + (env & ~1);
    double u0[4], u1[4], u2[4];
    stream_uniforms(RP.seed, gid, ep, 1, 0, u0);
    stream_uniforms(RP.seed, gid, ep, 1, 1, u1);
    stream_uniforms(RP.seed, gid, ep, 1, 2, u2);
    const float fix_spd = (float)(0.5 + 2.5 * u0[0]);
    const int wflag = (int)floor(2.0 * u0[1]);
    const double foot_mu = (double)P.fr_lo + u0[2] * ((double)P.fr_hi - (double)P.fr_lo);
    const double px = robot == 0 ? -2.0 + 4.0 * u0[3] : -2.0 + 4.0 * u1[1], py = robot == 0 ? -2.0 + 4.0 * u1[0] : -2.0 + 4.0 * u1[2];
    // both robots are handed the same mutable init dict => one running yaw for the pair (CTG:209-215)
    const double acc0 = E.aux[aux::yaw_accum_deg * N + (env & ~1)];
    const double yaw_a = fmod(acc0 + 360.0 * u1[3], 360.0), yaw_b = fmod(yaw_a + 360.0 * u2[0], 360.0);
    float q[3], qd[3];
    V3 lin, ang;
    const Q4 qn = start_pose(M, k, robot == 0 ? yaw_a : yaw_b, q, qd, lin, ang);
    const Q4 qI = base_qI(M);
    const Q4 qp = qmul(qnormalize(qn), qconj(qI));
    PairState PS = {robot == 0 ? wflag : 1 - wflag, 0, 1, 0, -2.0 + 4.0 * u2[1], -2.0 + 4.0 * u2[2]};
    // reset() runs _prepare_drill too (CTG:302): its flag-switch test reads the stale manifolds of the previous episode's last step
    const bool touch_own = E.aux[aux::flag_touch * N + env] != 0.0;
    float* snew = &s_new[threadIdx.x >> 2][0];
    const float* spart = &s_new[(threadIdx.x >> 2) ^ 1][0];
    sepmc_pair_tail(M, L, k, robot, snew, spart, px, py, 0.5, qp, qn, lin, ang, q, touch_own, fix_spd, RP.seed, gid, ep, PS);
#pragma unroll
    for (int i = 0; i < 3; i++) { snew[3 * k + i] = q[i]; snew[12 + 3 * k + i] = qd[i]; }
    int push_draws = 0;
    float pf[3] = {0.f, 0.f, 0.f};
    if (P.push_enabled) push_draws = 1;                              // PR:52-54: draw #0 becomes the current _randomized_force
    if (doit) {
      const V3 f = mul(qmat(qp), foot_in_base(L, q[0], q[1], q[2]));
      store_state(E, N, env, k, q, qd, V3{(float)px + f.x, (float)py + f.y, 0.5f + f.z}, px, py, 0.5, qn, lin, ang);
      E.warm[k * N + env] = 0.f;
      if (k == 0) {
        E.time[env] = 0.0; E.reward_sum[env] = 0.f; E.episode_steps[env] = 0; E.episode[env] = ep + 1;
        double* A = E.aux;
        A[aux::counter * N + env] = 0; A[aux::with_flag * N + env] = PS.with_flag; A[aux::flag_x * N + env] = PS.flag_x;
        A[aux::flag_y * N + env] = PS.flag_y; A[aux::control_spd * N + env] = fix_spd; A[aux::oppo_visible * N + env] = PS.visible;
        A[aux::switch_flag * N + env] = PS.sw; A[aux::total_spd * N + env] = 0.0; A[aux::max_spd * N + env] = 0.0;
        A[aux::push_count * N + env] = P.push_start_count;
        A[aux::push_fx * N + env] = pf[0]; A[aux::push_fy * N + env] = pf[1]; A[aux::push_fz * N + env] = pf[2];
        A[aux::foot_friction * N + env] = foot_mu; A[aux::push_draws * N + env] = push_draws; A[aux::flag_draws * N + env] = PS.flag_draws;
        A[aux::yaw_accum_deg * N + env] = yaw_b; A[aux::flag_touch * N + env] = touch_own ? 1.0 : 0.0;
      }
    }
  } else if (ENV == kEpmcFlat || ENV == kEpmcCorridor) {
    // ---------------- EPMC reset (PGE:196-249)
    long long ep = E.episode[env];
    const long long gid = RP.gid0 + env;
    double u[4];
    stream_uniforms(RP.seed, gid, ep, 1, 0, u);
    const double foot_mu = (double)P.fr_lo + u[0] * ((double)P.fr_hi - (double)P.fr_lo);                   // PGE:209-210
    int push_draws = 0;
    float pf[3] = {0.f, 0.f, 0.f};
    if (P.push_enabled) epmc_randomize_push(P, RP.seed, gid, ep, push_draws, pf);                          // PR:52-54
    const int cmd_freq = P.cmd_freq_lo + (int)floor(u[2] * (double)(P.cmd_freq_hi - P.cmd_freq_lo));       // PGE:223
    const double yaw_deg = fmod(E.aux[aux::yaw_accum_deg * N + env] + 360.0 * u[1], 360.0);                 // PGE:181-189 (accumulates)
    float q[3], qd[3];
    V3 lin, ang;
    const Q4 qn = start_pose(M, k, yaw_deg, q, qd, lin, ang);
    float* snew = &s_new[threadIdx.x >> 2][0];
    const M3 Rq = qmat(qnormalize(qn));
    const float target_spd = (float)E.aux[aux::target_spd * N + env];   // persists across episodes (PGE:170-172)
    double tgx0 = 8.0;
    int nb0 = 0;
    if (ENV == kEpmcCorridor) nb0 = generate_corridor(P, RP.seed, gid, ep, E.boxes + (size_t)env * (6 * kMaxBoxes), doit && k == 0, tgx0);   // PGE:216-219
#pragma unroll
    for (int i = 0; i < 3; i++) { snew[3 * k + i] = q[i]; snew[12 + 3 * k + i] = qd[i]; }
    // the tail's row at pos (0, 0, 0.5) with target (tgx0, 0); element 0: (8, 0) (BSE:247-248)
    if (k == 0) stage_epmc(snew, Rq, ang, lin, 0.0, 0.0, 0.5, tgx0, 0.0, target_spd);
    if (ENV == kEpmcCorridor) {
      __syncwarp();                                                 // lane 0's boxes are visible to the env's other lanes
      stage_corridor_masks(snew, E.boxes + (size_t)env * (6 * kMaxBoxes), doit ? nb0 : E.nbox[env], k, 0.f, 0.f, 0.5f, atan2f(Rq.a10, Rq.a00));
    }
    if (doit) {
      const Q4 qI = base_qI(M);
      const V3 f = mul(qmat(qmul(qnormalize(qn), qconj(qI))), foot_in_base(L, q[0], q[1], q[2]));
      E.warm[k * N + env] = 0.f;
      store_state(E, N, env, k, q, qd, V3{f.x, f.y, 0.5f + f.z}, 0.0, 0.0, 0.5, qn, lin, ang);
      if (k == 0) {
        E.time[env] = 0.0; E.reward_sum[env] = 0.f; E.episode_steps[env] = 0; E.episode[env] = ep + 1;
        double* A = E.aux;
        A[aux::counter * N + env] = 0; A[aux::cmd_vary_freq * N + env] = cmd_freq; A[aux::target_x * N + env] = tgx0;
        A[aux::target_y * N + env] = 0.0; A[aux::last_pos_diff_len * N + env] = fabs(tgx0); A[aux::total_spd * N + env] = 0.0;
        A[aux::init_pos_diff_len * N + env] = fabs(tgx0);                                                   // PGE:192-195
        if (ENV == kEpmcCorridor) E.nbox[env] = nb0;
        A[aux::max_spd * N + env] = 0.0; A[aux::push_count * N + env] = P.push_start_count;
        A[aux::push_fx * N + env] = pf[0]; A[aux::push_fy * N + env] = pf[1]; A[aux::push_fz * N + env] = pf[2];
        A[aux::foot_friction * N + env] = foot_mu; A[aux::push_draws * N + env] = push_draws; A[aux::cmd_draws * N + env] = 0;
        A[aux::yaw_accum_deg * N + env] = yaw_deg;
      }
    }
  } else {
  int clip; double t0;
  long long ep = E.episode[env];
  if (RP.mode == 2) {
    clip = RP.clip_in[env]; t0 = RP.time_in[env];
    if (!doit) { clip = 0; t0 = 0.0; }     // entries of masked-out envs are not validated by the host: never index the table with them
  } else {
    long long gid = RP.gid0 + env;
    unsigned c4[4] = {(unsigned)gid, (unsigned)((unsigned long long)gid >> 32), (unsigned)ep, (unsigned)((unsigned long long)ep >> 32)};
    philox4x32_10(c4, (unsigned)RP.seed, (unsigned)(RP.seed >> 32));
    double u1 = ((double)c4[0] + 0.5) * (1.0 / 4294967296.0), u2 = ((double)c4[1] + 0.5) * (1.0 / 4294967296.0);
    clip = C - 1;
    for (int c = 0; c < C; c++) if (s_cdf[c] > u1) { clip = c; break; }
    int nf = mc.clip_off[clip + 1] - mc.clip_off[clip];
    t0 = u2 * (P.frame_dt * (double)(nf - P.margin - 1));
    ep += 1;
  }
  int frame_id = (int)floor(t0 / P.frame_dt);
  double frac = (t0 - frame_id * P.frame_dt) / P.frame_dt;
  {
    const int last = mc.clip_off[clip + 1] - mc.clip_off[clip] - P.margin + 2;
    if (frame_id > last) { frame_id = last; frac = 0.0; }
    if (frame_id < 0) { frame_id = 0; frac = 0.0; }
  }
  const MocapFrame* f0 = mc.frames + mc.clip_off[clip] + frame_id;
  KinBase kb = mocap_base(f0, f0 + 1, frac, P.frame_dt);
  float inv = (float)(1.0 / P.frame_dt), fr = (float)frac;
  float q[3], qd[3];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    float c = f0->q[3 * k + i], n = f0[1].q[3 * k + i];
    q[i] = fmaf(fr, n - c, c);
    qd[i] = (n - c) * inv;
  }
  float* snew = &s_new[threadIdx.x >> 2][0];
  build_obs_new(mc, P, M, k, clip, frame_id, frac, kb.px, kb.py, kb.pz, kb.q, kb.lin, kb.ang, q, qd, snew);
  if (doit) {
    const Q4 qI = base_qI(M);
    const V3 f = mul(qmat(qmul(qnormalize(kb.q), qconj(qI))), foot_in_base(L, q[0], q[1], q[2]));
    store_state(E, N, env, k, q, qd, V3{(float)kb.px + f.x, (float)kb.py + f.y, (float)kb.pz + f.z}, kb.px, kb.py, kb.pz, kb.q, kb.lin, kb.ang);
#pragma unroll
    for (int i = 0; i < 3; i++) { E.kin[(state::q + 3 * k + i) * N + env] = q[i]; E.kin[(state::qd + 3 * k + i) * N + env] = qd[i]; }
    E.warm[k * N + env] = 0.f;
    if (k == 0) {
      const float b[10] = {kb.q.x, kb.q.y, kb.q.z, kb.q.w, kb.lin.x, kb.lin.y, kb.lin.z, kb.ang.x, kb.ang.y, kb.ang.z};   // quat | lin | ang
      E.kin[state::pos * N + env] = (float)kb.px; E.kin[(state::pos + 1) * N + env] = (float)kb.py; E.kin[(state::pos + 2) * N + env] = (float)kb.pz;
#pragma unroll
      for (int i = 0; i < 10; i++) E.kin[(state::quat + i) * N + env] = b[i];
      E.time[env] = t0; E.clip[env] = clip; E.reward_sum[env] = 0.f; E.episode_steps[env] = 0; E.episode[env] = ep;
      E.ob_id[env] = 0;                                            // PLE:179
    }
  }
  }
  __syncwarp();
  unsigned rows = 0;
#pragma unroll
  for (int e = 0; e < 8; e++) if ((wm >> (4 * e)) & 1u) rows |= 1u << e;
  const int warp_env0 = (blockIdx.x * BLOCK + (threadIdx.x & ~31)) >> 2;
  emit_obs_rows<ENV>(E.obs, obs2, obs2_ld, &s_new[(threadIdx.x & ~31) >> 2][0], &s_new[0][0], warp_env0, N, 1, rows, E.boxes);
}

}  // namespace llq
