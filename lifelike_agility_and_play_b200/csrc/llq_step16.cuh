// llq_step16.cuh -- the fused policy-step kernel, 16 lanes per environment (DESIGN.md 2, 4.1).
//
// Mapping: one environment = one half-warp.  Lane l (0..15) of the half-warp plays three roles during a 2 ms sub-step:
//   * link lane   leg k = l & 3, link i = l >> 2 (0 hip, 1 thigh, 2 shank; i = 3: the base body): rigid-body inertia and bias
//                 wrench of ONE body in base coordinates -> composite inertias (suffix sums along the leg) -> its column F_i of the
//                 base/joint coupling block and its row of the leg's 3x3 joint-space inertia H_k (composite-rigid-body form);
//   * sphere lane collision spheres l and l + 16 of the robot (feet, knee wheels, hips, thighs, shanks, trunk corners) against
//                 the ground / arena walls / corridor boxes, compacted into the env's contact list with one ballot;
//   * row lane    ONE constraint row of the sub-step's LCP: its image (y, w) under the block factorisation of the mass matrix, its row
//                 of Delassus coefficients (shared memory) and its impulse in Bullet's sequential-impulse sweep, where every row
//                 update is one __shfl_sync broadcast + one FMA per lane.  For this role the CTA's envs are re-paired by row count
//                 every sub-step (heaviest with lightest) and the rows of a pair are packed into the warp's 32 lanes -- a lane's row
//                 may belong to either env of the pair, or (after the re-pairing) to an env another warp owns (see solve_rows).
// The dynamics are the same equations Bullet's articulated-body algorithm solves, factorised block-wise instead of link by link:
//   [ Ic  F ] [a0]   [-p0   ]        H_k = L D L^T per leg,  S = Ic - sum_k F_k H_k^-1 F_k^T = L0 L0^T  (6x6, replicated),
//   [ F^T H ] [qdd] = [tau - C]       J M^-1 J'^T = y.y' + [same leg] w.(D^-1 w'),  y = L0^-1 (G - F_k H_k^-1 j),  w = L^-1 j.
// Everything is expressed in base coordinates about the base reference point (an inertial frame that coincides with the base at
// the start of the sub-step), so composite inertias and bias wrenches simply add.
//
// Replaces the same reference calls as llq_kernels.cuh's header lists (PLE:195-245, LR:119-148, stepSimulation, ML:65-166).
#pragma once
#include "llq_kernels.cuh"

namespace llq {

#ifndef LLQ16_BLOCK
#define LLQ16_BLOCK 224   // 14 envs per CTA: 4096 envs = 293 CTAs = one wave of 2 CTAs (14 warps) per SM; 256 would put 16 warps on 108 of the
                          // 148 SMs (0.263 -> 0.247 ms); 128 / 160 threads: 0.256 / 0.249 ms (DESIGN.md 4.1)
#endif
#ifndef LLQ16_MINB
#define LLQ16_MINB 4   // resident CTAs per SM the register budget is sized for (4 x 128 threads x 128 registers = the whole file)
#endif
constexpr int kMaxSph = 32, kMaxCon = 8, kMaxLim = 8;
struct SphConst { float c[3]; float r; float mu_link; int leg; int depth; int foot; };   // centre in the frame of link (leg, depth - 1); depth 0 = base
struct alignas(16) SphTable { int n; int rule; int pad[2]; SphConst s[kMaxSph]; };         // rule: llq_config.knee_contacts

// ---- per-env shared-memory tables (floats): one block of kEnvFloats per env, split into six tables by env_tabs
// link record 3 k + i (link i of leg k): its rotation Rx(c1, s1) Ry(cy, sy) and origin p in base coordinates
namespace linkrec { constexpr int c1 = 0, s1 = 1, cy = 2, sy = 3, p = 4, end = 7; }
constexpr int kLinkW = 8, kLinkTab = 12 * kLinkW;
// leg table of leg k, in two layouts.  Dynamics phase: column F_i of the coupling block (angular 3 | linear 3) at F + 6 i, row i of H_k
// at H + 3 i, the joints' right-hand sides, and the leg's composite mass, first moment, inertia (xx xy xz yy yz zz) and bias wrench
// (angular 3 | linear 3).  Rows phase, from the end of the forward dynamics on: column m of W = F L^-T at W + 6 m, L (L10 L20 L21),
// D^-1, the predicted joint velocities, and the knee joint's c3, s3 for the fp64 clearance of the shank's spheres.
namespace legdyn { constexpr int F = 0, H = 18, rhs = 27, m = 30, h = 31, Ic = 34, bias = 40, end = 46; }
namespace legrow { constexpr int W = 0, L = 18, dinv = 21, qd = 24, c3 = 28, s3 = 29, end = 30; }
constexpr int kLegW = 48, kLegTab = 4 * kLegW;
static_assert(legdyn::end <= kLegW && legrow::end <= kLegW, "each phase of the leg table fits its 48 floats");
// contact record: leg (-1: the base) and depth of the sphere's link (int bits), contact point, normal n and tangents t1 t2 (base
// coordinates), clearance, friction, warm-start impulse, final normal impulse
namespace conrec { constexpr int leg = 0, depth = 1, Pc = 2, n = 5, t1 = 8, t2 = 11, dist = 14, mu = 15, lam0 = 16, lam = 17, end = 18; }
constexpr int kConW = 20, kConTab = kMaxCon * kConW;
static_assert(conrec::t1 == conrec::n + 3 && conrec::t2 == conrec::n + 6, "row_image reads direction d at n + 3 d");
static_assert(conrec::depth == conrec::leg + 1 && conrec::Pc == conrec::depth + 1 && conrec::n == conrec::Pc + 3 && conrec::dist == conrec::t2 + 3 &&
              conrec::mu == conrec::dist + 1 && conrec::leg % 4 == 0 && conrec::end <= kConW && kConW % 4 == 0,
              "the contact writer stores leg .. mu as four float4");
// limit row: leg, joint (int bits), direction, penetration
namespace limrec { constexpr int leg = 0, joint = 1, dir = 2, pen = 3; }
constexpr int kLimW = 4, kLimTab = kMaxLim * kLimW;
static_assert(limrec::joint == limrec::leg + 1 && limrec::dir == limrec::leg + 2 && limrec::pen == limrec::leg + 3 && limrec::leg == 0,
              "the limit writer stores a row as one float4");
// constraint row: its image y, e = D^-1 w and leg (int bits), for the other rows' Delassus entries
namespace rowrec { constexpr int y = 0, e = 6, leg = 9; }
constexpr int kRowW = 12, kRowTab = 32 * kRowW;
static_assert(rowrec::y == 0 && rowrec::e == rowrec::y + 6 && rowrec::leg == rowrec::e + 3 && kRowW == 12,
              "rows are moved as three float4: y0-3 | y4 y5 e0 e1 | e2 leg - -");
// The row table's storage is also, in turn: the dynamics phase's scratch (one record of kScrW floats per lane), the solver's totals
// (the impulse sums: base 6, then 3 per leg) and the hand-over to the step tail (TailState).
constexpr int kScrW = 20;
static_assert(16 * kScrW <= kRowTab, "the dynamics scratch lives in the row table");
namespace sums { constexpr int base = 0, leg = 6, end = 18; }
static_assert(sums::leg == sums::base + 6 && sums::end == sums::leg + 3 * 4 && sums::end <= kRowTab, "the impulse sums live in the row table");
// env table: the base body's bias wrench (dynamics), which then becomes the predicted base velocity (rows) | packed Cholesky factor of
// the base block | joint targets | actions
namespace envslot { constexpr int bias = 0, vel = 0, chol = 8, target = 32, act = 44; }
constexpr int kEnvTab = 56;
static_assert(envslot::bias + 6 <= envslot::chol && envslot::chol + 21 <= envslot::target && envslot::target + kActDim <= envslot::act &&
              envslot::act + kActDim <= kEnvTab, "env table slots");
constexpr int kEnvFloats = 944;        // >= the sum of the tables, and = 16 (mod 32): envs an odd number of slots apart hit disjoint banks
static_assert(kLinkTab + kLegTab + kConTab + kLimTab + kRowTab + kEnvTab <= kEnvFloats && kEnvFloats % 32 == 16, "per-env table layout");
struct EnvTabs { float *link, *leg, *con, *lim, *row, *env; };
LLQ_DI EnvTabs env_tabs(float* block) {          // block = s_env_dyn + e * kEnvFloats
  EnvTabs t;
  t.link = block; t.leg = t.link + kLinkTab; t.con = t.leg + kLegTab; t.lim = t.con + kConTab; t.row = t.lim + kLimTab; t.env = t.row + kRowTab;
  return t;
}
// Delassus coefficients of one WARP (its two envs' rows packed into 32 lanes): column col of lane l at col * stride + l.  Contact c,
// direction d -> column con + 3 c + d; limit row t -> column lim + t.
namespace dcol { constexpr int con = 0, lim = 3 * kMaxCon, n = lim + kMaxLim, stride = 32; }
constexpr int kATabWarp = dcol::n * dcol::stride;
// staging-row borrows before the tail: the corridor's candidate boxes (6 floats each) and the SEPMC proxy points of each leg (foot |
// knee wheel | hip | two body corners | handle, 3 floats each)
constexpr int kProxyW = 18;
static_assert(6 * kMaxCand <= kNewObs && 4 * kProxyW <= kNewObs, "the candidate boxes and the proxy points fit a staging row");

LLQ_DI V3 rotxy(V3 v, float cy, float sy, float cx, float sx) { return rot<0>(rot<1>(v, cy, sy), cx, sx); }     // Rx Ry v
LLQ_DI V3 rotxyT(V3 v, float cy, float sy, float cx, float sx) { return rotT<1>(rotT<0>(v, cx, sx), cy, sy); }  // (Rx Ry)^T v
LLQ_DI float dot6(const float (&a)[6], const float (&b)[6]) {
  return fmaf(a[0], b[0], fmaf(a[1], b[1], fmaf(a[2], b[2], fmaf(a[3], b[3], fmaf(a[4], b[4], a[5] * b[5])))));
}
// rigid-body inertia about the base origin from the one about the link origin at p (h' = rotated first moment)
LLQ_DI Sym3 shift_inertia(Sym3 I, float m, V3 h, V3 p) {
  const float ph = dot(p, h);
  Sym3 o;
  o.xx = I.xx + m * (p.y * p.y + p.z * p.z) + 2.f * (ph - p.x * h.x);
  o.yy = I.yy + m * (p.x * p.x + p.z * p.z) + 2.f * (ph - p.y * h.y);
  o.zz = I.zz + m * (p.x * p.x + p.y * p.y) + 2.f * (ph - p.z * h.z);
  o.xy = I.xy - m * p.x * p.y - (p.x * h.y + h.x * p.y);
  o.xz = I.xz - m * p.x * p.z - (p.x * h.z + h.x * p.z);
  o.yz = I.yz - m * p.y * p.z - (p.y * h.z + h.y * p.z);
  return o;
}
// bias wrench v x* (I v) of a body (m, h, I about the base origin, base axes) + Bullet's per-URDF-link damping, items given in the
// body's own link frame (rotation Rx(cx,sx) Ry(cy,sy), origin po)
LLQ_DI SV bias_wrench(float m, V3 h, Sym3 I, int nd, const DampItem* d, V3 w, V3 v, float kl, float ka, float cy, float sy, float cx, float sx, V3 po) {
  const V3 hl = fma3(m, v, cross(w, h));
  const V3 ha = mul(I, w) + cross(h, v);
  SV p;
  p.a = cross(w, ha) + cross(v, hl);
  p.l = cross(w, hl);
  const float wn = norm3(w);
  const V3 wl = rotxyT(w, cy, sy, cx, sx);
#pragma unroll
  for (int t = 0; t < 3; t++) {
    if (t < nd) {
      const V3 c = rotxy(ld3(d[t].c), cy, sy, cx, sx) + po;
      const V3 vc = v + cross(w, c);
      const V3 f = (d[t].m * (kl + kl * norm3(vc))) * vc;
      const V3 n = (ka + ka * wn) * rotxy(mul(ldsym(d[t].Ic), wl), cy, sy, cx, sx);
      p.l = p.l + f;
      p.a = p.a + n + cross(c, f);
    }
  }
  return p;
}
// triangular solves with the packed Cholesky factor (llq_math.cuh layout) kept in shared memory
LLQ_DI void chol6_fwd_p(const float* l, const float (&b)[6], float (&y)[6]) {
#pragma unroll
  for (int i = 0; i < 6; i++) {
    float s = b[i];
#pragma unroll
    for (int k = 0; k < i; k++) s = fmaf(-l[tri(i, k)], y[k], s);
    y[i] = s * l[tri(i, i)];
  }
}
LLQ_DI void chol6_bwd_p(const float* l, const float (&y)[6], float (&x)[6]) {
#pragma unroll
  for (int i = 5; i >= 0; i--) {
    float s = y[i];
#pragma unroll
    for (int k = i + 1; k < 6; k++) s = fmaf(-l[tri(k, i)], x[k], s);
    x[i] = s * l[tri(i, i)];
  }
}
LLQ_DI float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
LLQ_DI void st4(float* p, float a, float b, float c, float d) { *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d); }

// fp64 distance of a sphere centre (world) to an axis-aligned box (centre + half extents), with the contact normal (EPMC corridor)
LLQ_DI void sphere_box(double wx, double wy, double wz, double r, const float* b, double& db, V3& nn) {
  const double p0 = wx - (double)b[0], p1 = wy - (double)b[1], p2 = wz - (double)b[2];
  const double h0 = b[3], h1 = b[4], h2 = b[5];
  const double c0 = fmin(fmax(p0, -h0), h0), c1 = fmin(fmax(p1, -h1), h1), c2 = fmin(fmax(p2, -h2), h2);
  if (c0 != p0 || c1 != p1 || c2 != p2) {
    const double v0 = p0 - c0, v1 = p1 - c1, v2 = p2 - c2;
    const double len = sqrt(v0 * v0 + v1 * v1 + v2 * v2);
    db = len - r;
    nn = V3{(float)(v0 / len), (float)(v1 / len), (float)(v2 / len)};
  } else {                                 // centre inside the box: leave through the nearest face
    double best = h0 - p0; nn = V3{1.f, 0.f, 0.f};
    if (h0 + p0 < best) { best = h0 + p0; nn = V3{-1.f, 0.f, 0.f}; }
    if (h1 - p1 < best) { best = h1 - p1; nn = V3{0.f, 1.f, 0.f}; }
    if (h1 + p1 < best) { best = h1 + p1; nn = V3{0.f, -1.f, 0.f}; }
    if (h2 - p2 < best) { best = h2 - p2; nn = V3{0.f, 0.f, 1.f}; }
    if (h2 + p2 < best) { best = h2 + p2; nn = V3{0.f, 0.f, -1.f}; }
    db = -best - r;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Constraint rows of one sub-step for the warp's two envs: row images, Delassus rows, Bullet's sequential-impulse sweep
// (btMultiBodyConstraintSolver::solveSingleIteration order: limits, normals, friction pairs with the implicit cone).
//
// One row per lane, the rows of the two envs PACKED into the warp's 32 lanes: env A (the lower half-warp's) owns lanes [0, split),
// env B lanes [split, 32); an env's rows are its contacts' (3 per contact: normal, two tangents), then its limit rows.  split = 16
// whenever both envs have <= 16 rows; an env with more borrows lanes of its partner (3 c + l <= 32 rows per env by the caps); a pair
// with more than 32 rows between them is solved in two passes, each env on all 32 lanes.  A lane therefore reads the tables of the env
// its ROW belongs to (RowsIn::tb), which need not be the env its link / sphere roles belong to.  The Delassus coefficients of a row
// live in shared memory (atab[col * 32 + lane], col = position of the other row in its env's row list: conflict free); all loops are
// rolled, with warp-uniform bounds, and indexed by per-lane owners -- the whole solver is ~300 instructions of code.
// The warp's two envs are ANY two envs of the CTA (the kernel pairs heavy with light ones after a CTA barrier); the totals
// sum lam_r y_r (base part, 6) and, per leg, sum lam_r w_r (joint part, 4 x 3) go back through the env's row table.
// ---- development aid (-DLLQ16_TIMING, tools/warp_timing.py): per-warp clock64 totals of the sub-step phases
#ifdef LLQ16_TIMING
__device__ unsigned long long g_t16[16384 * 12];
#define T16_DECL long long t16_[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, t16_c = clock64(), t16_s = t16_c
#define T16_MARK(slot) { const long long t16_n = clock64(); t16_[slot] += t16_n - t16_c; t16_c = t16_n; }
#define T16_ADD(slot, v) t16_[slot] += (v)
#define T16_IN(slot) { const long long t16_n = clock64(); in.t16[slot] += t16_n - *in.t16c; *in.t16c = t16_n; }
#else
#define T16_DECL
#define T16_MARK(slot)
#define T16_ADD(slot, v)
#define T16_IN(slot)
#endif
struct RowsIn {
#ifdef LLQ16_TIMING
  long long* t16; long long* t16c;
#endif
  float* tb;            // table block (s_env_dyn + e * kEnvFloats) of the env this lane's ROW belongs to
  float* acol;          // this lane's column of the warp's coefficient table: acol[col * 32]
  int nc, nl;           // contacts / limit rows of that env
  int rr;               // index of this lane's row in the env's row list (>= 3 nc + nl: no row)
  int lane0;            // first lane of that env's rows
  int lane;             // 0..31
  int split;            // warp-uniform: 16 = every row on its own env's half-warp
  int Cmax, Lmax;       // warp-uniform maxima over the envs of this pass: contacts, limit rows
  float* res;           // where the totals of the env behind this lane's HALF-warp go (the impulse sums, at the head of its row table), or
                        // nullptr when that env is not solved in this pass
  float dt, slop, erp, jerp, max_imp;
  int iters;
};
// one row: its image under the factorised mass matrix and the scalars of the sweep
struct RowRegs { float y[6], wj[3], b, rhs, invd, lam, hi, mu; int leg; };
// row rr of the env behind in.tb: contact rr / 3 in direction rr % 3, or limit row rr - 3 nc; also leaves (y, e = D^-1 w, leg) in the
// env's row table for the other rows' Delassus entries.  Returns true for a normal row (its impulse is the contact's warm start).
LLQ_DI bool row_image(const RowsIn& in, RowRegs& r) {
  const EnvTabs tab = env_tabs(in.tb);
  const int rr = in.rr;
  const bool is_con = rr < 3 * in.nc;
  const int d = rr % 3, cq = rr / 3;
  float e[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int t = 0; t < 6; t++) r.y[t] = 0.f;
  r.wj[0] = r.wj[1] = r.wj[2] = 0.f;
  r.b = 0.f; r.rhs = 0.f; r.invd = 0.f; r.lam = 0.f; r.hi = 0.f; r.mu = 0.f; r.leg = -2;
  const bool act = rr < 3 * in.nc + in.nl;
  if (act) {
    V3 Ga = V3{0.f, 0.f, 0.f}, Gl = V3{0.f, 0.f, 0.f};
    float j[3] = {0.f, 0.f, 0.f}, rel = 0.f, dist = 0.f, lam0 = 0.f, pen = 0.f, dirl = 0.f;
    int leg, jj = 0;
    if (is_con) {
      const float* cr = tab.con + cq * kConW;
      leg = __float_as_int(cr[conrec::leg]);
      const int depth = __float_as_int(cr[conrec::depth]);
      const V3 Pc = ld3(cr + conrec::Pc), dir = ld3(cr + conrec::n + 3 * d);
      dist = cr[conrec::dist]; r.mu = cr[conrec::mu]; lam0 = cr[conrec::lam0];
      Ga = cross(Pc, dir); Gl = dir;
      // predicted base velocity (base coordinates), parked by the env's lane 0
      rel = dot(Ga, ld3(tab.env + envslot::vel)) + dot(Gl, ld3(tab.env + envslot::vel + 3));
      if (leg >= 0) {
        const float* lk = tab.link + 3 * leg * kLinkW;     // links 0, 1, 2 of the leg
        const float c1 = lk[linkrec::c1], s1 = lk[linkrec::s1];
        const V3 p1 = ld3(lk + linkrec::p), p2 = ld3(lk + kLinkW + linkrec::p), p3 = ld3(lk + 2 * kLinkW + linkrec::p), n2 = V3{0.f, -c1, -s1};
        j[0] = Ga.x + dot(cross(p1, V3{1.f, 0.f, 0.f}), Gl);
        if (depth >= 2) j[1] = dot(n2, Ga) + dot(cross(p2, n2), Gl);
        if (depth >= 3) j[2] = dot(n2, Ga) + dot(cross(p3, n2), Gl);
      }
    } else {
      const float* lr = tab.lim + (rr - 3 * in.nc) * kLimW;
      leg = __float_as_int(lr[limrec::leg]); jj = __float_as_int(lr[limrec::joint]); dirl = lr[limrec::dir]; pen = lr[limrec::pen];
      j[0] = jj == 0 ? dirl : 0.f; j[1] = jj == 1 ? dirl : 0.f; j[2] = jj == 2 ? dirl : 0.f;
    }
    r.leg = leg;
    float g[6] = {Ga.x, Ga.y, Ga.z, Gl.x, Gl.y, Gl.z};
    if (leg >= 0) {
      const float* lt = tab.leg + leg * kLegW;
      const float L10 = lt[legrow::L], L20 = lt[legrow::L + 1], L21 = lt[legrow::L + 2];
      rel += j[0] * lt[legrow::qd] + j[1] * lt[legrow::qd + 1] + j[2] * lt[legrow::qd + 2];
      r.wj[0] = j[0];
      r.wj[1] = fmaf(-L10, r.wj[0], j[1]);
      r.wj[2] = fmaf(-L20, r.wj[0], fmaf(-L21, r.wj[1], j[2]));
      e[0] = r.wj[0] * lt[legrow::dinv]; e[1] = r.wj[1] * lt[legrow::dinv + 1]; e[2] = r.wj[2] * lt[legrow::dinv + 2];
#pragma unroll
      for (int m = 0; m < 3; m++)
#pragma unroll
        for (int t = 0; t < 6; t++) g[t] = fmaf(-e[m], lt[legrow::W + 6 * m + t], g[t]);
    }
    chol6_fwd_p(tab.env + envslot::chol, g, r.y);
    const float dg = dot6(r.y, r.y) + r.wj[0] * e[0] + r.wj[1] * e[1] + r.wj[2] * e[2];
    r.invd = 1.0f / dg;
    if (is_con) {
      if (d == 0) {   // btMultiBodyConstraintSolver::setupMultiBodyContactConstraint
        const float pn = dist + in.slop;
        float poserr = 0.f, velerr = -rel;
        if (pn > 0.f) velerr -= pn / in.dt; else poserr = -pn * in.erp / in.dt;
        r.rhs = (poserr + velerr) * r.invd;
        r.lam = lam0; r.hi = 1e10f;
      } else {
        r.rhs = -rel * r.invd;
      }
    } else {
      const float poserr = pen > -0.04f ? -pen * in.jerp / in.dt : 0.f;   // split-impulse threshold quirk (SURVEY A.2c)
      r.rhs = (poserr - rel) * r.invd;
      r.hi = in.max_imp;
    }
    float* rw = tab.row + rr * kRowW + rowrec::y;
    st4(rw, r.y[0], r.y[1], r.y[2], r.y[3]);
    st4(rw + 4, r.y[4], r.y[5], e[0], e[1]);
    st4(rw + 8, e[2], __int_as_float(r.leg), 0.f, 0.f);
  }
  return act && is_con && d == 0;
}
// entry (r, col) of the Delassus matrix from this lane's row r and the table entry of row `col`
LLQ_DI float delassus_entry(const RowRegs& r, const float* rw) {
  const float4 a = ld4(rw), bq = ld4(rw + 4), cq4 = ld4(rw + 8);
  const float ys[6] = {a.x, a.y, a.z, a.w, bq.x, bq.y};
  const float jt = r.wj[0] * bq.z + r.wj[1] * bq.w + r.wj[2] * cq4.x;
  return dot6(r.y, ys) + (__float_as_int(cq4.y) == r.leg ? jt : 0.f);
}
// total impulse of an env: Yt += sum lam_r y_r and, per leg, sum lam_r w_r -- 18 values.  Rows that sit on the partner's half-warp are
// handed across first (xor 16), then a butterfly over each half-warp.
LLQ_DI void impulse_sums(const RowsIn& in, const RowRegs& r) {
  float v18[sums::end];
#pragma unroll
  for (int t = 0; t < 6; t++) v18[sums::base + t] = r.lam * r.y[t];
#pragma unroll
  for (int kk = 0; kk < 4; kk++) {
    const float f = r.leg == kk ? r.lam : 0.f;
#pragma unroll
    for (int m = 0; m < 3; m++) v18[sums::leg + 3 * kk + m] = f * r.wj[m];
  }
  if (in.split != 16) {                                     // warp-uniform
    const bool foreign = (in.lane >= 16) != (in.lane >= in.split);      // the row belongs to the other half-warp's env
#pragma unroll
    for (int t = 0; t < sums::end; t++) {                   // (unrolled: a rolled loop would index v18 in local memory)
      const float mine = foreign ? 0.f : v18[t], give = foreign ? v18[t] : 0.f;
      v18[t] = mine + __shfl_xor_sync(FULL, give, 16);
    }
  }
#pragma unroll 1
  for (int o = 1; o < 16; o <<= 1) {
#pragma unroll
    for (int t = 0; t < sums::end; t++) v18[t] += __shfl_xor_sync(FULL, v18[t], o);
  }
  if (in.res && (in.lane & 15) == 0) {                    // the lower half-warp holds env A's totals, the upper one env B's
#pragma unroll
    for (int t = 0; t + 4 <= sums::end; t += 4) st4(in.res + t, v18[t], v18[t + 1], v18[t + 2], v18[t + 3]);
#pragma unroll
    for (int t = sums::end & ~3; t < sums::end; t++) in.res[t] = v18[t];
  }
}

LLQ_DI void solve_rows(const RowsIn& in) {
  int lane = in.lane;
  asm volatile("" : "+r"(lane));            // opaque: held in a register instead of being re-derived from %tid at every row
  RowRegs r;
  const bool is_normal = row_image(in, r);
  __syncwarp();
  T16_IN(8);
  float* acol = in.acol;
  const int lane0 = in.lane0, nc = in.nc, nl = in.nl;
  // Coefficient columns (dcol): contact c, direction d -> column con + 3 c + d; limit row t -> column lim + t.  Columns the sweep visits
  // for the partner's sake (its lists are longer) hold zeros, so that those steps change nothing; the loop bounds are rounded up to
  // even (the sweeps are unrolled by two; the caps are even).
  const int Ce = (in.Cmax + 1) & ~1, Le = (in.Lmax + 1) & ~1;
  {
    const float* rowtab = env_tabs(in.tb).row;
    const int ncon = 3 * nc;
#pragma unroll 1
    for (int col = 0; col < 3 * Ce; col++) {
      const float a = delassus_entry(r, rowtab + col * kRowW);
      acol[(dcol::con + col) * dcol::stride] = col < ncon ? a : 0.f;        // (beyond the env's list the table holds old rows: finite, masked)
    }
    const float* rl = rowtab + ncon * kRowW;
#pragma unroll 1
    for (int t = 0; t < Le; t++) {
      const float a = delassus_entry(r, rl + t * kRowW);
      acol[(dcol::lim + t) * dcol::stride] = t < nl ? a : 0.f;
    }
  }
  // warm start of the normal rows
#pragma unroll 1
  for (int c = 0; c < in.Cmax; c++) r.b = fmaf(acol[(dcol::con + 3 * c) * dcol::stride], __shfl_sync(FULL, r.lam, lane0 + 3 * c), r.b);
  T16_IN(9);
  // projected Gauss-Seidel (btMultiBodyConstraintSolver::solveSingleIteration order).  One row update: candidate on every lane (only
  // the owner's counts), owner commits, broadcast, one LDS + FMA per lane.  Dependent chain per row: FFMA (candidate from
  // c = lam + rhs, kept up to date off the chain) -> 2 FMNMX -> FADD -> SHFL -> FFMA.
  float rc = r.lam + r.rhs;
#define LLQ16_CLAMP_LIMIT(x) fminf(fmaxf((x), 0.f), r.hi)      /* joint-limit rows: [0, max impulse] */
#define LLQ16_CLAMP_NORMAL(x) fmaxf((x), 0.f)                  /* normal rows: [0, 1e10] -- the upper bound never binds a finite state */
#define LLQ16_ROW_UPDATE(src, a, valid, CLAMP)                                                        \
  {                                                                                                   \
    const float cl = CLAMP(fmaf(-r.b, r.invd, rc));      /* clamp the accumulated impulse */           \
    const float dl = cl - r.lam;                                                                      \
    const bool own = lane == (src) && (valid);                                                        \
    r.lam = own ? cl : r.lam;                                                                         \
    rc = own ? cl + r.rhs : rc;                                                                       \
    r.b = fmaf((a), __shfl_sync(FULL, dl, (src)), r.b);                                               \
  }
#pragma unroll 1
  for (int it = 0; it < in.iters; it++) {
    {
      int src = lane0 + 3 * nc;
      const float* ap = acol + dcol::lim * dcol::stride;
#pragma unroll 1
      for (int t = 0; t < Le; t += 2, src += 2, ap += 2 * dcol::stride) {     // joint-limit rows in joint order
        LLQ16_ROW_UPDATE(src, ap[0], t < nl, LLQ16_CLAMP_LIMIT)
        LLQ16_ROW_UPDATE(src + 1, ap[dcol::stride], t + 1 < nl, LLQ16_CLAMP_LIMIT)
      }
    }
    {
      int src = lane0;
      const float* ap = acol + dcol::con * dcol::stride;
#pragma unroll 1
      for (int t = 0; t < Ce; t += 2, src += 6, ap += 6 * dcol::stride) {    // normal rows in contact order
        LLQ16_ROW_UPDATE(src, ap[0], t < nc, LLQ16_CLAMP_NORMAL)
        LLQ16_ROW_UPDATE(src + 3, ap[3 * dcol::stride], t + 1 < nc, LLQ16_CLAMP_NORMAL)
      }
    }
    {
      int src = lane0;
      const float* ap = acol + dcol::con * dcol::stride;
#pragma unroll 1
      for (int t = 0; t < in.Cmax; t++, src += 3, ap += 3 * dcol::stride) {   // friction pairs with the implicit cone (resolveConeFrictionConstraintRows)
        // One shuffle round trip on the dependent chain: the two tangent rows' candidates go to every lane together with their current
        // impulses and the cone's radius (those three do not depend on this step's b), and every lane forms both increments itself.
        const float sown = fmaf(-r.b, r.invd, rc);
        const float sa = __shfl_sync(FULL, sown, src + 1), sb = __shfl_sync(FULL, sown, src + 2);
        const float la = __shfl_sync(FULL, r.lam, src + 1), lb = __shfl_sync(FULL, r.lam, src + 2);
        const float limit = __shfl_sync(FULL, r.mu * r.lam, src);
        const float r2 = sa * sa + sb * sb;
        const float rs = rsqrtf(r2);                           // issued before the comparison resolves (inf for r2 = 0: not selected)
        const bool clip = r2 >= limit * limit && r2 > 0.f;
        const float sc = limit * rs;
        const float na = clip ? sa * sc : sa, nb = clip ? sb * sc : sb;
        const bool valid = t < nc;
        if (lane == src + 1 && valid) { r.lam = na; rc = na + r.rhs; }
        if (lane == src + 2 && valid) { r.lam = nb; rc = nb + r.rhs; }
        r.b = fmaf(ap[dcol::stride], na - la, fmaf(ap[2 * dcol::stride], nb - lb, r.b));
      }
    }
  }
#undef LLQ16_ROW_UPDATE
#undef LLQ16_CLAMP_LIMIT
#undef LLQ16_CLAMP_NORMAL
  T16_IN(10);
  // the normal impulses go back to the contact records (warm start of the next sub-step)
  if (is_normal) env_tabs(in.tb).con[(in.rr / 3) * kConW + conrec::lam] = r.lam;
  __syncwarp();                     // every lane is done with the row table: its head becomes the result area
  impulse_sums(in, r);
}

// ---------------------------------------------------------------------------------------------------------------
// End of the policy step: observation, reward, termination, write-back -- run by FOUR lanes per env (lane k = leg k, 8 envs per
// warp) on the first EPB / 8 warps of the CTA, from the state the sub-step lanes left in shared memory.  With 16 lanes per env this
// part (mocap interpolation, four future targets, reward, the cooperative emission of the observation rows) would run once per TWO
// envs; here one instruction stream serves eight.
struct TailState {            // per env, written by the env's lane 0 (base part) and its lanes (k, 0) (joint part)
  double px, py, pz, time, frame_frac;
  int frame_id, ob_id, flags, push_count, push_draws;      // flags: tflag bits
  float pf[3], qp[4], vw[3], ww[3], q[12], qd[12];
};
namespace tflag { constexpr int bad = 1, ob_hit = 2, touch_own = 4, tag = 8; }
static_assert(sizeof(TailState) <= sizeof(float) * kRowTab, "the hand-over record lives in the row table");
template <int ENV>
LLQ_DI void step_tail(const EnvArrays& E, const MocapDev& mc, const StepParams& P, const ModelConst& M, float* s_new, const float* s_hist,
                      const TailState& T, const float* act_src, float* obs2, long long obs2_ld, int* winner, unsigned long long seed, long long gid0,
                      int record, int el, int k, int env, bool valid) {
  const int N = P.n_envs;
  double px = T.px, py = T.py, pz = T.pz, time = T.time, frame_frac = T.frame_frac;
  int frame_id = T.frame_id, ob_id = T.ob_id, push_count = T.push_count, push_draws = T.push_draws;
  bool bad = (T.flags & tflag::bad) != 0, ob_hit = (T.flags & tflag::ob_hit) != 0;
  const bool touch_own = (T.flags & tflag::touch_own) != 0, tag = (T.flags & tflag::tag) != 0;
  const float pf[3] = {T.pf[0], T.pf[1], T.pf[2]};
  const Q4 qp = Q4{T.qp[0], T.qp[1], T.qp[2], T.qp[3]};
  const V3 vw = V3{T.vw[0], T.vw[1], T.vw[2]}, ww = V3{T.ww[0], T.ww[1], T.ww[2]};
  float q[3], qd[3];
#pragma unroll
  for (int t = 0; t < 3; t++) { q[t] = T.q[3 * k + t]; qd[t] = T.qd[3 * k + t]; }
  const int clip = ENV == kPmc ? E.clip[env] : 0;
  const long long epi = ENV != kPmc ? E.episode[env] - 1 : 0;
  const int robot = env & 1;
  const long long pair_gid = gid0 + (env & ~1);
  bool done = false;
  float rew_out = 0.f;
  const bool wr = valid;
  const LegConst& L = M.leg[k];
  const Q4 qI = Q4{M.base.qI[0], M.base.qI[1], M.base.qI[2], M.base.qI[3]};
  Q4 qb;
  PairState PS = {0, 0, 1, 0, 0.0, 0.0};
  if (ENV == kPmc) {
    qb = qmul(qp, qI);                                 // back to the pybullet (inertial-frame) convention
    float* snew = s_new + el * kNewObs;
    ObsCtx oc = build_obs_new(mc, P, M, k, clip, frame_id, frame_frac, px, py, pz, qb, vw, ww, q, qd, snew);
#pragma unroll
    for (int t = 0; t < 3; t++) snew[kPropDim + 3 * k + t] = act_src[3 * k + t];
    // reward (PLE:350-426)
    float djp = 0.f, djv = 0.f;
#pragma unroll
    for (int t = 0; t < 3; t++) { float a = q[t] - oc.kq[t], b = qd[t] - oc.kqd[t]; djp = fmaf(a, a, djp); djv = fmaf(b, b, djv); }
    V3 fd, fk;
    {
      M3 Rp = qmat(qp);
      V3 f = mul(Rp, foot_in_base(L, q[0], q[1], q[2]));
      fd = V3{(float)px + f.x, (float)py + f.y, (float)pz + f.z};
      Q4 kqp = qmul(qnormalize(oc.kb.q), qconj(qI));
      V3 g = mul(qmat(kqp), foot_in_base(L, oc.kq[0], oc.kq[1], oc.kq[2]));
      // difference of foot positions, formed in double for the base offset
      fk = V3{(float)(oc.kb.px - px) + g.x - f.x, (float)(oc.kb.py - py) + g.y - f.y, (float)(oc.kb.pz - pz) + g.z - f.z};
    }
    float dee = dot(fk, fk);
    djp = gsum4(djp); djv = gsum4(djv); dee = gsum4(dee);
    float dpx = (float)(px - oc.kb.px), dpy = (float)(py - oc.kb.py), dpz = (float)(pz - oc.kb.pz);
    float dp = dpx * dpx + dpy * dpy + dpz * dpz;
    V3 dvl3 = vw - oc.kb.lin, dva3 = ww - oc.kb.ang;
    Q4 q1 = qnormalize(qb), q2 = qnormalize(oc.kb.q);
    float angle = norm3(q_rotvec(qnormalize(qmul(q2, qconj(q1)))));
    float rew = P.w_jp * expf(-1.0f * djp) + P.w_jv * expf(-0.1f * djv) + P.w_ee * expf(-40.0f * dee) +
                P.w_pose * expf(-20.0f * dp - 10.0f * angle * angle) + P.w_vel * expf(-2.0f * dot(dvl3, dvl3) - 0.2f * dot(dva3, dva3));
    // termination (PLE:337-348, LR:158-179, ML:168-172)
    bool fall = fallen(qmat(q1));
    int nf = mc.clip_off[clip + 1] - mc.clip_off[clip];
    bool ended = frame_id >= nf - P.margin - 1;
    bool diff = fabsf(angle) > 1.0f || dp > 1.0f;
    if (bad || !isfinite(rew)) { rew = 0.f; bad = true; }
    if (P.has_ob) {
      int oh = ob_hit ? 1 : 0;
      oh |= __shfl_xor_sync(FULL, oh, 1);
      oh |= __shfl_xor_sync(FULL, oh, 2);
      ob_hit = oh != 0;
      const int o0 = mc.ob_off[clip], n_ob = mc.ob_off[clip + 1] - o0;                 // PLE:262-268 hand-over to the next plate
      while (ob_id < n_ob - 1 && time > mc.ob_table[(size_t)(o0 + ob_id) * 4] + 0.5) ob_id++;
    }
    done = fall || ended || diff || ob_hit || bad;                                     // PLE:347
    rew_out = rew;
    if (wr) {
      store_state(E, N, env, k, q, qd, fd, px, py, pz, qb, vw, ww);
#pragma unroll
      for (int t = 0; t < 3; t++) { E.kin[(state::q + 3 * k + t) * N + env] = oc.kq[t]; E.kin[(state::qd + 3 * k + t) * N + env] = oc.kqd[t]; }
      if (k == 0) {
        if (P.has_ob) E.ob_id[env] = ob_id;
        E.kin[state::pos * N + env] = (float)oc.kb.px; E.kin[(state::pos + 1) * N + env] = (float)oc.kb.py; E.kin[(state::pos + 2) * N + env] = (float)oc.kb.pz;
        E.kin[state::quat * N + env] = oc.kb.q.x; E.kin[(state::quat + 1) * N + env] = oc.kb.q.y;
        E.kin[(state::quat + 2) * N + env] = oc.kb.q.z; E.kin[(state::quat + 3) * N + env] = oc.kb.q.w;
        E.kin[state::lin * N + env] = oc.kb.lin.x; E.kin[(state::lin + 1) * N + env] = oc.kb.lin.y; E.kin[(state::lin + 2) * N + env] = oc.kb.lin.z;
        E.kin[state::ang * N + env] = oc.kb.ang.x; E.kin[(state::ang + 1) * N + env] = oc.kb.ang.y; E.kin[(state::ang + 2) * N + env] = oc.kb.ang.z;
        if (done) {
          E.done_reward[env] = E.reward_sum[env] + rew;
          atomicMax(&winner[clip], env);       // highest finished env index owns the clip's slot this step (PLE:236)
        }
      }
    }
  } else if (ENV == kSepmc) {
    // ---------------- SEPMC tail (CTG:378-424, 458-470, 495-596, 640-652)
    const double* A = E.aux;
    int counter = (int)A[aux::counter * N + env];
    PS.with_flag = (int)A[aux::with_flag * N + env]; PS.flag_x = A[aux::flag_x * N + env]; PS.flag_y = A[aux::flag_y * N + env];
    const float fix_spd = (float)A[aux::control_spd * N + env];
    double total_spd = A[aux::total_spd * N + env], max_spd = A[aux::max_spd * N + env];
    PS.flag_draws = (int)A[aux::flag_draws * N + env];
    qb = qmul(qp, qI);
    float* snew = s_new + el * kNewObs;
    const float* spart = s_new + (el ^ 1) * kNewObs;
    sepmc_pair_tail(M, L, k, robot, snew, spart, px, py, pz, qp, qb, vw, ww, q, touch_own, fix_spd, seed, pair_gid, epi, PS);
#pragma unroll
    for (int t = 0; t < 3; t++) { snew[3 * k + t] = q[t]; snew[12 + 3 * k + t] = qd[t]; snew[kPropDim + 3 * k + t] = act_src[3 * k + t]; }
    const float spd = sqrtf(vw.x * vw.x + vw.y * vw.y);              // stat_spd (CTG:368-373)
    total_spd += (double)spd;
    if ((double)spd > max_spd) max_spd = (double)spd;
    counter += 1;
    int fall = fallen(qmat(qnormalize(qb))) ? 1 : 0;
    const int fall_other = __shfl_xor_sync(FULL, fall, 4);
    if (robot == 1) fall = fall_other;                                  // only robot 0's fall ends the episode (CTG:462)
    bad = bad || __shfl_xor_sync(FULL, bad ? 1 : 0, 4) != 0;
    done = fall != 0 || counter >= P.max_steps || tag || bad;
    // rewards (CTG:640-652, 412-419): +-1 on a flag switch, +-1 on a tag; with_flag after the switch
    const int wf0 = robot == 0 ? PS.with_flag : 1 - PS.with_flag;       // does robot 0 hold the flag
    float rew = (float)PS.sw * ((wf0 != 0) == (robot == 0) ? 1.f : -1.f);
    if (done && tag) rew += (wf0 != 0) == (robot == 0) ? 1.f : -1.f;
    if (bad) rew = 0.f;
    rew_out = rew;
    if (wr) {
      const V3 f = mul(qmat(qp), foot_in_base(L, q[0], q[1], q[2]));
      store_state(E, N, env, k, q, qd, V3{(float)px + f.x, (float)py + f.y, (float)pz + f.z}, px, py, pz, qb, vw, ww);
      if (k == 0) {
        double* Aw = E.aux;
        Aw[aux::counter * N + env] = counter; Aw[aux::with_flag * N + env] = PS.with_flag; Aw[aux::flag_x * N + env] = PS.flag_x;
        Aw[aux::flag_y * N + env] = PS.flag_y; Aw[aux::oppo_visible * N + env] = PS.visible; Aw[aux::switch_flag * N + env] = PS.sw;
        Aw[aux::total_spd * N + env] = total_spd; Aw[aux::max_spd * N + env] = max_spd; Aw[aux::push_count * N + env] = push_count;
        Aw[aux::push_fx * N + env] = pf[0]; Aw[aux::push_fy * N + env] = pf[1]; Aw[aux::push_fz * N + env] = pf[2];
        Aw[aux::push_draws * N + env] = push_draws; Aw[aux::flag_draws * N + env] = PS.flag_draws;
        Aw[aux::flag_touch * N + env] = touch_own ? 1.0 : 0.0;
      }
    }
  } else {
    // ---------------- EPMC tail (PGE:302-321, 334-358, 360-372, 479-539)
    const double* A = E.aux;
    int counter = (int)A[aux::counter * N + env], cmd_draws = (int)A[aux::cmd_draws * N + env];
    const int cmd_freq = (int)A[aux::cmd_vary_freq * N + env];
    double tgx = A[aux::target_x * N + env], tgy = A[aux::target_y * N + env], target_angle = A[aux::target_angle * N + env];
    double last_len = A[aux::last_pos_diff_len * N + env];
    double total_spd = A[aux::total_spd * N + env], max_spd = A[aux::max_spd * N + env];
    float target_spd = (float)A[aux::target_spd * N + env];
    const double init_len = ENV == kEpmcCorridor ? A[aux::init_pos_diff_len * N + env] : 1.0;
    {
      // the command of this step was drawn from the pose at the START of the step (PGE:302-317): recover it from the stored state
      const double sx0 = E.pos[env], sy0 = E.pos[N + env];
      if (counter % cmd_freq == 0) {
        double uu[4];
        stream_uniforms(seed, gid0 + env, epi, 3, (unsigned)cmd_draws++, uu);
        if (ENV == kEpmcFlat) {
          target_angle = 2.0 * 3.14159265358979323846 * uu[0];
          double sn, cs;
          sincos(target_angle, &sn, &cs);
          tgx = sx0 + cs * 100.0; tgy = sy0 + sn * 100.0;
          last_len = sqrt((sx0 - tgx) * (sx0 - tgx) + (sy0 - tgy) * (sy0 - tgy));
        }
        target_spd = (float)((double)P.ts_lo + uu[1] * ((double)P.ts_hi - (double)P.ts_lo));
      }
      if (ENV == kEpmcCorridor) target_angle = atan2(tgy - sy0, tgx - sx0);     // PGE:318-323 (plotting only)
    }
    __syncwarp();                                        // the pose above is read before lane 0 overwrites it below
    qb = qmul(qp, qI);
    float* snew = s_new + el * kNewObs;
    const Q4 q1 = qnormalize(qb);
    const M3 Rq = qmat(q1);
#pragma unroll
    for (int t = 0; t < 3; t++) { snew[3 * k + t] = q[t]; snew[12 + 3 * k + t] = qd[t]; snew[kPropDim + 3 * k + t] = act_src[3 * k + t]; }
    counter += 1;
    const double dx = tgx - px, dy = tgy - py;
    const double plen = sqrt(dx * dx + dy * dy);
    if (k == 0) stage_epmc(snew, Rq, ww, vw, px, py, pz, dx, dy, target_spd);
    const bool fall = fallen(Rq);
    const bool reach = plen < 0.5, timeup = counter >= P.max_steps;
    const float ux = (float)(dx / plen), uy = (float)(dy / plen);
    const float spd = fabsf(vw.x * ux + vw.y * uy);
    total_spd += (double)spd;
    if ((double)spd > max_spd) max_spd = (double)spd;
    const float yaw = atan2f(Rq.a10, Rq.a00);
    float sy_, cy_;
    llq_sincosf(yaw, &sy_, &cy_);
    float rew = expf(-fabsf(spd - target_spd)) * expf((cy_ * ux + sy_ * uy - 1.0f) * 5.0f) / (float)P.max_steps;
    if (ENV == kEpmcCorridor) {                                        // _compute_avg_spd_reward (PGE:504-539)
      const float reward_rot = expf((cy_ * ux + sy_ * uy - 1.0f) * 5.0f);
      const float reward_dist = (float)((plen - last_len) / init_len);
      last_len = plen;
      rew = reward_rot / (float)P.max_steps * 0.1f * 2.0f - reward_dist * 0.1f;
      if (reach) rew += expf(-fabsf((float)(total_spd / (double)counter) - target_spd));
      stage_corridor_masks(snew, E.boxes + (size_t)env * (6 * kMaxBoxes), E.nbox[env], k, (float)px, (float)py, (float)pz, yaw);
    }
    if (bad || !isfinite(rew)) { rew = 0.f; bad = true; }
    done = fall || timeup || reach || bad;
    rew_out = rew;
    if (wr) {
      const V3 f = mul(qmat(qp), foot_in_base(L, q[0], q[1], q[2]));
      store_state(E, N, env, k, q, qd, V3{(float)px + f.x, (float)py + f.y, (float)pz + f.z}, px, py, pz, qb, vw, ww);
      if (k == 0) {
        double* Aw = E.aux;
        Aw[aux::counter * N + env] = counter; Aw[aux::cmd_vary_freq * N + env] = cmd_freq; Aw[aux::target_x * N + env] = tgx;
        Aw[aux::target_y * N + env] = tgy; Aw[aux::target_spd * N + env] = target_spd; Aw[aux::target_angle * N + env] = target_angle;
        Aw[aux::last_pos_diff_len * N + env] = last_len; Aw[aux::total_spd * N + env] = total_spd; Aw[aux::max_spd * N + env] = max_spd;
        Aw[aux::push_count * N + env] = push_count;
        Aw[aux::push_fx * N + env] = pf[0]; Aw[aux::push_fy * N + env] = pf[1]; Aw[aux::push_fz * N + env] = pf[2];
        Aw[aux::push_draws * N + env] = push_draws; Aw[aux::cmd_draws * N + env] = cmd_draws;
      }
    }
  }
  if (wr && k == 0) {                                    // end-of-step bookkeeping of every level
    E.time[env] = time;
    E.reward_sum[env] += rew_out;
    E.episode_steps[env] += 1;
    E.reward[env] = rew_out;
    E.done[env] = done ? 1 : 0;
  }
  // record mode (llq_set_option "record"): the trajectory columns action 12 | reward | done behind the observation of the slab row;
  // record == 2: into the slab row before the one that receives the observation (parallel/rollout.py)
  if (record && obs2 && wr) {
    float* row = obs2 + (size_t)env * obs2_ld + ObsW<ENV>::value - (record == 2 ? (long long)N * obs2_ld : 0ll);
#pragma unroll
    for (int t = 0; t < 3; t++) row[3 * k + t] = act_src[3 * k + t];
    if (k == 0) { row[kRecReward] = rew_out; row[kRecDone] = done ? 1.f : 0.f; }
  }
  {
    const unsigned dm = __ballot_sync(FULL, valid && k == 0 && done);       // episodes finished: one atomic per warp
    if ((threadIdx.x & 31) == 0 && dm) atomicAdd(&E.counters[1], (unsigned long long)__popc(dm));
  }
  // (the observation rows are emitted by ALL warps of the CTA after a barrier: kernel epilogue)
}

// ---------------------------------------------------------------------------------------------------------------
template <int ENV>
__global__ void __launch_bounds__(LLQ16_BLOCK, LLQ16_MINB * 128 / LLQ16_BLOCK) llq_step16_kernel(EnvArrays E, MocapDev mc, StepParams P, const ModelConst* __restrict__ gmodel,
                                                            const SphTable* __restrict__ gsph, const float* __restrict__ actions,
                                                            float* obs2, long long obs2_ld, int* __restrict__ winner,
                                                            unsigned long long seed, long long gid0, int record) {
  constexpr int BLOCK = LLQ16_BLOCK, EPB = BLOCK / 16;        // 2 envs per warp
  constexpr int EPT = (EPB + 7) / 8 * 8;                      // the tail runs 8 envs per warp on whole warps: rows EPB.. are dummies
  static_assert(BLOCK % 32 == 0 && EPB <= 32, "whole warps; one lane per env in the pairing");
  __shared__ __align__(16) ModelConst M;
  __shared__ __align__(16) SphTable ST;
  __shared__ __align__(16) float s_new[EPT][kNewObs];
  __shared__ __align__(16) float s_hist[EPT][kHist];
  __shared__ int s_cnt[32];                                   // contacts | limit rows << 8 of the CTA's envs, this sub-step
  extern __shared__ __align__(16) float s_env_dyn[];   // [EPB][kEnvFloats] per-env tables, then one kATabWarp coefficient table per warp
  const int tid = threadIdx.x;
  const int N = P.n_envs;
  prefetch_model(gmodel, &M, BLOCK);
  {
    const float4* src = reinterpret_cast<const float4*>(gsph);
    float4* dst = reinterpret_cast<float4*>(&ST);
    for (int t = tid; t < (int)(sizeof(SphTable) / 16); t += BLOCK) __pipeline_memcpy_async(dst + t, src + t, 16);
  }
  __pipeline_commit();
  const int warp_env0 = blockIdx.x * EPB + ((tid >> 5) << 1);
  prefetch_history<ENV, 2>(E.obs, &s_hist[(tid >> 5) << 1][0], warp_env0, N);
  __pipeline_commit();
  __pipeline_wait_prior(1);              // model constants have landed; the history copy stays in flight
  __syncthreads();

  const int l16 = tid & 15, k = l16 & 3, i = l16 >> 2, el = tid >> 4;
  const int env_raw = blockIdx.x * EPB + el;
  const int env = env_raw < N ? env_raw : N - 1;   // surplus lanes shadow the last env (they must join the shuffles)
  const bool valid = env_raw < N;
  const LegConst& L = M.leg[k];
  const V3 r0 = ld3(L.j[0].r), r1 = ld3(L.j[1].r), r2 = ld3(L.j[2].r);
  // this env's tables, the env_tabs split spelled out: taking the same pointers from an EnvTabs changes ptxas's schedule of this kernel
  float* const linktab = s_env_dyn + el * kEnvFloats;
  float* const legtab = linktab + kLinkTab;
  float* const contab = legtab + kLegTab;
  float* const limtab = contab + kConTab;
  float* const rowtab = limtab + kLimTab;
  float* const scr = rowtab;                         // dynamics-phase scratch (16 lanes x kScrW floats) aliases the row table
  float* const envtab = rowtab + kRowTab;
  float* const s_atab = s_env_dyn + EPB * kEnvFloats;   // [BLOCK / 32][dcol::n][32 lanes] Delassus coefficients, one table per warp
  for (int col = 0; col < dcol::n; col++) s_atab[(tid >> 5) * kATabWarp + col * dcol::stride + (tid & 31)] = 0.f;      // finite from the start (masked steps multiply them by 0)
  // joints with a lower dof index than this lane's (k, i): rank of a violated limit in Bullet's row order
  unsigned lowmask = 0;
#pragma unroll
  for (int t = 0; t < 12; t++) if (3 * (t & 3) + (t >> 2) < 3 * k + i) lowmask |= 1u << t;

  // ---- load state (base entries replicated on the 16 lanes, joint entries on the 4 lanes of the leg)
  double px = E.pos[env], py = E.pos[N + env], pz = E.pos[2 * N + env];
  const float* sr = E.st;
  Q4 qb = Q4{sr[st::quat * N + env], sr[(st::quat + 1) * N + env], sr[(st::quat + 2) * N + env], sr[(st::quat + 3) * N + env]};
  V3 vw = V3{sr[st::lin * N + env], sr[(st::lin + 1) * N + env], sr[(st::lin + 2) * N + env]};
  V3 ww = V3{sr[st::ang * N + env], sr[(st::ang + 1) * N + env], sr[(st::ang + 2) * N + env]};
  float q[3], qd[3];
#pragma unroll
  for (int t = 0; t < 3; t++) {
    q[t] = sr[(st::q + 3 * k + t) * N + env];
    qd[t] = sr[(st::qd + 3 * k + t) * N + env];
  }
  if (i < 3) {                                               // joint (k, i): action and clipped target stay in shared memory
    const float a = actions[(size_t)env * kActDim + 3 * k + i];
    envtab[envslot::act + 3 * k + i] = a;
    envtab[envslot::target + 3 * k + i] = clampf((i == 0 ? q[0] : (i == 1 ? q[1] : q[2])) + a, -3.0f, 3.0f);           // PLE:200, LR:126-127
  }
  const int nsph = ST.n, rule = ST.rule;
  float warm[2];                                             // remembered normal impulses of spheres l16 and l16 + 16
  warm[0] = l16 < nsph ? E.warm[(size_t)l16 * N + env] : 0.f;
  warm[1] = 16 + l16 < nsph ? E.warm[(size_t)(16 + l16) * N + env] : 0.f;
  double time = E.time[env];
  const int clip = ENV == kPmc ? E.clip[env] : 0;
  int frame_id = 0; double frame_frac = 0.0;
  int ob_id = 0; bool ob_hit = false;
  if (ENV == kPmc && P.has_ob) ob_id = E.ob_id[env];
  // ---- EPMC / SEPMC bookkeeping used inside the sub-steps (the rest is read in the tail)
  int push_count = 0, push_draws = 0;
  float pf[3] = {0.f, 0.f, 0.f}, mu_env = P.mu;
  long long epi = 0;
  PairState PS = {0, 0, 1, 0, 0.0, 0.0};
  bool touch_own = false, tag = false;
  const int robot = env & 1;
  const long long pair_gid = gid0 + (env & ~1);
  if (ENV != kPmc) {
    const double* A = E.aux;
    push_count = (int)A[aux::push_count * N + env];
    pf[0] = (float)A[aux::push_fx * N + env]; pf[1] = (float)A[aux::push_fy * N + env]; pf[2] = (float)A[aux::push_fz * N + env];
    mu_env = P.mu_ground * (float)A[aux::foot_friction * N + env]; push_draws = (int)A[aux::push_draws * N + env];
    epi = E.episode[env] - 1;                             // streams of the running episode (the reset advanced the counter)
    if (ENV == kSepmc) { PS.flag_x = A[aux::flag_x * N + env]; PS.flag_y = A[aux::flag_y * N + env]; }
  }
  // ---- EPMC corridor: the boxes the robot can reach during this step -> shared memory (<= kMaxCand per env)
  int n_cand = 0;
  float* s_cand = nullptr;
  if (ENV == kEpmcCorridor) {
    s_cand = &s_new[el][0];                            // the staging row is free until the tail: kMaxCand x 6 floats
    const float* bxs = E.boxes + (size_t)env * (6 * kMaxBoxes);
    // reach of the robot's spheres from the base reference point: hip offset 0.195 + leg 0.48 in x, 0.15 + 0.05 in y, plus the
    // travel during the step (<= 0.06 m at 3 m/s) -> 0.8 m per axis (0.6 missed hind feet stretched backwards over a hurdle)
    unsigned long long m = box_mask(bxs, E.nbox[env], k, (float)px, (float)py, (float)pz, 0.8f, false);
    int c = 0;
    while (m && c < kMaxCand) {
      const int j = __ffsll((long long)m) - 1;
      m &= m - 1;
      if ((c & 3) == k && i == 0) {
#pragma unroll
        for (int t = 0; t < 6; t++) s_cand[6 * c + t] = bxs[6 * j + t];
      }
      c++;
    }
    n_cand = c;
    __syncwarp();
  }
  // base orientation: pybullet speaks in the base inertial frame; dynamics run in URDF body axes B' = inertial * qI^-1
  const Q4 qI = base_qI(M);
  Q4 qp = qmul(qnormalize(qb), qconj(qI));
  unsigned n_contact_rows = 0, n_limit_rows = 0, n_overflow = 0;
  bool bad = false;
  const float mu_foot = ENV != kPmc ? mu_env : P.mu;

  T16_DECL;
  for (int sub = 0; sub < P.substeps; sub++) {
    T16_MARK(5);
    const float dt = P.dt;
    // ---------------- push randomiser (PR:56-87): counters in sub-steps, force lasts one sub-step
    bool push_on = false;
    if (ENV == kSepmc && P.push_enabled) {
      push_count += 1;
      if (push_count > 0) {
        if (push_count % P.push_interval == 0) { push_draws += 1; push_count = 0; }
        if (push_count < P.push_duration) {
          int draw = push_draws - 1 + robot;
          epmc_randomize_push(P, seed, pair_gid, epi, draw, pf);
          push_draws += 2;
          push_on = true;
        }
      }
    }
    if ((ENV == kEpmcFlat || ENV == kEpmcCorridor) && P.push_enabled) {
      push_count += 1;
      if (push_count > 0) {
        if (push_count % P.push_interval == 0) { epmc_randomize_push(P, seed, gid0 + env, epi, push_draws, pf); push_count = 0; }
        push_on = push_count < P.push_duration;
      }
    }
    V3 wbs, vbs;                                  // predicted base velocity in base coordinates (the rows' generalised velocity)
    {   // ================ forward dynamics; everything declared here dies at the closing brace (register budget of the solver)
    // ---------------- kinematics: every lane evaluates the sine / cosine of its own joint, the leg's six values go round by shuffle
    const M3 R = qmat(qp);                       // world <- B'
    float c1, s1, c2, s2, c3, s3;
    {
      float so, co;
      llq_sincosf(i == 0 ? q[0] : (i == 1 ? -q[1] : -q[2]), &so, &co);
      c1 = __shfl_sync(FULL, co, k, 16); s1 = __shfl_sync(FULL, so, k, 16);
      c2 = __shfl_sync(FULL, co, k + 4, 16); s2 = __shfl_sync(FULL, so, k + 4, 16);
      c3 = __shfl_sync(FULL, co, k + 8, 16); s3 = __shfl_sync(FULL, so, k + 8, 16);
    }
    const float c23 = c2 * c3 - s2 * s3, s23 = s2 * c3 + c2 * s3;
    const V3 p1 = r0;
    const V3 p2 = p1 + rot<0>(r1, c1, s1);
    const V3 p3 = p2 + rot<0>(rot<1>(r2, c2, s2), c1, s1);
    const V3 n2 = V3{0.f, -c1, -s1};                                       // axis of joints 2, 3 (= -E1 e_y)
    // this lane's body: rotation Rx(cx, sx) Ry(cy, sy), origin po (the base body: identity, 0)
    const float cx = i == 3 ? 1.f : c1, sx = i == 3 ? 0.f : s1;
    const float cy = i == 1 ? c2 : (i == 2 ? c23 : 1.f), sy = i == 1 ? s2 : (i == 2 ? s23 : 0.f);
    const V3 po = i == 0 ? p1 : (i == 1 ? p2 : (i == 2 ? p3 : V3{0.f, 0.f, 0.f}));
    const V3 wb = tmul(R, ww), vb = tmul(R, vw);     // base velocity, base coordinates
    // ---------------- velocity and velocity-product acceleration of the body (joints below it contribute nothing)
    const V3 l1 = cross(p1, V3{1.f, 0.f, 0.f}), l2 = cross(p2, n2), l3 = cross(p3, n2);
    SV v = SV{wb, vb}, ab = SV{V3{0.f, 0.f, 0.f}, V3{0.f, 0.f, 0.f}};
    {
      const float e0 = i < 3 ? qd[0] : 0.f, e1 = (i == 1 || i == 2) ? qd[1] : 0.f, e2 = i == 2 ? qd[2] : 0.f;
      V3 ja = V3{e0, 0.f, 0.f}, jl = e0 * l1;
      v.a = v.a + ja; v.l = v.l + jl;
      ab.a = cross(v.a, ja); ab.l = cross(v.a, jl) + cross(v.l, ja);
      ja = e1 * n2; jl = e1 * l2;
      v.a = v.a + ja; v.l = v.l + jl;
      ab.a = ab.a + cross(v.a, ja); ab.l = ab.l + cross(v.a, jl) + cross(v.l, ja);
      ja = e2 * n2; jl = e2 * l3;
      v.a = v.a + ja; v.l = v.l + jl;
      ab.a = ab.a + cross(v.a, ja); ab.l = ab.l + cross(v.a, jl) + cross(v.l, ja);
    }
    // ---------------- rigid-body inertia about the base origin and bias wrench of the body
    const int ic = i < 3 ? i : 0;
    const float bm_ = i == 3 ? M.base.m : L.j[ic].m;
    const float* hp = i == 3 ? M.base.h : L.j[ic].h;
    const float* Ip = i == 3 ? M.base.I : L.j[ic].I;
    const DampItem* dp = i == 3 ? M.base.d : L.j[ic].d;
    const int nd = i == 3 ? M.base.nd : L.j[ic].nd;
    const V3 hr = rotxy(ld3(hp), cy, sy, cx, sx);
    const Sym3 Ir = rot_sym<0>(rot_sym<1>(ldsym(Ip), cy, sy), cx, sx);
    V3 hc = fma3(bm_, po, hr);
    Sym3 Ic = shift_inertia(Ir, bm_, hr, po);
    float mc_ = bm_;
    SV f = bias_wrench(bm_, hc, Ic, nd, dp, v.a, v.l, P.kl, P.ka, cy, sy, cx, sx, po);
    f.a = f.a + mul(Ic, ab.a) + cross(hc, ab.l);
    f.l = f.l + bm_ * ab.l + cross(ab.a, hc);
    if (ENV != kPmc && push_on && l16 == 0) {
      // applyExternalForce(link 0 = FR hip, LINK_FRAME): force given in the hip's inertial frame, applied at its CoM (PR:73-77)
      const V3 fl = V3{M.push_R[0] * pf[0] + M.push_R[1] * pf[1] + M.push_R[2] * pf[2], M.push_R[3] * pf[0] + M.push_R[4] * pf[1] + M.push_R[5] * pf[2],
                       M.push_R[6] * pf[0] + M.push_R[7] * pf[1] + M.push_R[8] * pf[2]};
      const V3 fb_ = rot<0>(fl, c1, s1), cb_ = rot<0>(ld3(M.push_c), c1, s1) + p1;
      f.a = f.a - cross(cb_, fb_);
      f.l = f.l - fb_;
    }
    // ---------------- composite inertia / accumulated bias wrench along the leg (suffix sums through the scratch rows)
    {
      float* my = scr + l16 * kScrW;
      st4(my, f.a.x, f.a.y, f.a.z, f.l.x); st4(my + 4, f.l.y, f.l.z, mc_, hc.x);
      st4(my + 8, hc.y, hc.z, Ic.xx, Ic.xy); st4(my + 12, Ic.xz, Ic.yy, Ic.yz, Ic.zz);
      __syncwarp();
      if (i < 2) {
#pragma unroll 1
        for (int up = i + 1; up < 3; up++) {
          const float* o = scr + (k + 4 * up) * kScrW;
          const float4 a = ld4(o), b4 = ld4(o + 4), c4 = ld4(o + 8), d4 = ld4(o + 12);
          f.a = f.a + V3{a.x, a.y, a.z}; f.l = f.l + V3{a.w, b4.x, b4.y};
          mc_ += b4.z; hc = hc + V3{b4.w, c4.x, c4.y};
          Ic = Ic + Sym3{c4.z, c4.w, d4.x, d4.y, d4.z, d4.w};
        }
      }
    }
    // ---------------- this joint's column of the coupling block, its row of H_k, its right-hand side (PD torque, LR:138-141)
    {
      const V3 ax = i == 0 ? V3{1.f, 0.f, 0.f} : n2, al = cross(po, ax);
      const V3 Fa = mul(Ic, ax) + cross(hc, al), Fl = fma3(mc_, al, cross(ax, hc));
      const float Cb = dot(ax, f.a) + dot(al, f.l);
      const float h0 = Fa.x + dot(l1, Fl), h1 = dot(n2, Fa) + dot(l2, Fl), h2 = dot(n2, Fa) + dot(l3, Fl);
      const float qi = i == 0 ? q[0] : (i == 1 ? q[1] : q[2]), qdi = i == 0 ? qd[0] : (i == 1 ? qd[1] : qd[2]);
      const float tg = envtab[envslot::target + 3 * k + ic];
      const float tau = clampf(fmaf(P.kp, tg - qi, P.kd * (0.f - qdi)), -P.max_tau, P.max_tau) - L.j[ic].jdamp * qdi;
      float* lt = legtab + k * kLegW;
      if (i < 3) {
        float* Fi = lt + legdyn::F + 6 * i;
        Fi[0] = Fa.x; Fi[1] = Fa.y; Fi[2] = Fa.z; Fi[3] = Fl.x; Fi[4] = Fl.y; Fi[5] = Fl.z;
        lt[legdyn::H + 3 * i] = h0; lt[legdyn::H + 3 * i + 1] = h1; lt[legdyn::H + 3 * i + 2] = h2;
        lt[legdyn::rhs + i] = tau - Cb;
        float* lk = linktab + (3 * k + i) * kLinkW;
        st4(lk + linkrec::c1, c1, s1, cy, sy); st4(lk + linkrec::p, po.x, po.y, po.z, 0.f);
        if (i == 0) {
          lt[legdyn::m] = mc_; lt[legdyn::h] = hc.x; lt[legdyn::h + 1] = hc.y; lt[legdyn::h + 2] = hc.z;
          float* Il = lt + legdyn::Ic;
          Il[0] = Ic.xx; Il[1] = Ic.xy; Il[2] = Ic.xz; Il[3] = Ic.yy; Il[4] = Ic.yz; Il[5] = Ic.zz;
          float* bw = lt + legdyn::bias;
          bw[0] = f.a.x; bw[1] = f.a.y; bw[2] = f.a.z; bw[3] = f.l.x; bw[4] = f.l.y; bw[5] = f.l.z;
        }
      } else if (k == 0) {
        float* bw = envtab + envslot::bias;
        bw[0] = f.a.x; bw[1] = f.a.y; bw[2] = f.a.z; bw[3] = f.l.x; bw[4] = f.l.y; bw[5] = f.l.z;
      }
    }
    __syncwarp();
    // ---------------- per leg (replicated on its 4 lanes): H_k = L D L^T, Schur complement and right-hand side of the base
    float W[3][6], L10, L20, L21, di[3], u[3];
    float m6[21], z0[6];
    {
      const float* lt = legtab + k * kLegW;
#pragma unroll
      for (int m = 0; m < 3; m++)
#pragma unroll
        for (int t = 0; t < 6; t++) W[m][t] = lt[legdyn::F + 6 * m + t];
      const float* H = lt + legdyn::H;                     // row i at 3 i
      const float H00 = H[0], H10 = H[3], H11 = H[4], H20 = H[6], H21 = H[7], H22 = H[8];
      di[0] = 1.0f / H00;
      L10 = H10 * di[0]; L20 = H20 * di[0];
      const float d1 = fmaf(-L10, H10, H11);
      di[1] = 1.0f / d1;
      L21 = fmaf(-L20, H10, H21) * di[1];
      const float d2 = fmaf(-L20, H20, fmaf(-L21 * L21, d1, H22));
      di[2] = 1.0f / d2;
      // W = F L^-T (columns w_m), u = L^-1 rhs
#pragma unroll
      for (int t = 0; t < 6; t++) {
        W[1][t] = fmaf(-L10, W[0][t], W[1][t]);
        W[2][t] = fmaf(-L20, W[0][t], fmaf(-L21, W[1][t], W[2][t]));
      }
      const float* rhs = lt + legdyn::rhs;
      u[0] = rhs[0]; u[1] = fmaf(-L10, u[0], rhs[1]); u[2] = fmaf(-L20, u[0], fmaf(-L21, u[1], rhs[2]));
      const float cm = lt[legdyn::m];
      const V3 ch_ = ld3(lt + legdyn::h);
      const M3 hx = skew(ch_);
      const float* Il = lt + legdyn::Ic;                   // xx xy xz yy yz zz
      // packed lower triangle of [[A, B], [B^T, C]] : rows 0-2 = A, rows 3-5 = [B^T, C]
      m6[tri(0, 0)] = Il[0]; m6[tri(1, 0)] = Il[1]; m6[tri(1, 1)] = Il[3];
      m6[tri(2, 0)] = Il[2]; m6[tri(2, 1)] = Il[4]; m6[tri(2, 2)] = Il[5];
      m6[tri(3, 0)] = hx.a00; m6[tri(3, 1)] = hx.a10; m6[tri(3, 2)] = hx.a20;
      m6[tri(4, 0)] = hx.a01; m6[tri(4, 1)] = hx.a11; m6[tri(4, 2)] = hx.a21;
      m6[tri(5, 0)] = hx.a02; m6[tri(5, 1)] = hx.a12; m6[tri(5, 2)] = hx.a22;
      m6[tri(3, 3)] = cm; m6[tri(4, 3)] = 0.f; m6[tri(4, 4)] = cm; m6[tri(5, 3)] = 0.f; m6[tri(5, 4)] = 0.f; m6[tri(5, 5)] = cm;
#pragma unroll
      for (int m = 0; m < 3; m++) {
        const float ud = u[m] * di[m];
#pragma unroll
        for (int r = 0; r < 6; r++) {
          const float wd = W[m][r] * di[m];
#pragma unroll
          for (int c = 0; c <= r; c++) m6[tri(r, c)] = fmaf(-wd, W[m][c], m6[tri(r, c)]);
        }
#pragma unroll
        for (int t = 0; t < 6; t++) z0[t] = (m == 0 ? lt[legdyn::bias + t] : z0[t]) + ud * W[m][t];
      }
      // the four legs (xor 1, 2 stay inside the group of lanes with the same link index)
#pragma unroll
      for (int t = 0; t < 21; t++) m6[t] = gsum4(m6[t]);
#pragma unroll
      for (int t = 0; t < 6; t++) z0[t] = gsum4(z0[t]);
      const V3 bh = ld3(M.base.h); const Sym3 bI = ldsym(M.base.I); const float bm = M.base.m;
      const M3 bx = skew(bh);
      m6[tri(0, 0)] += bI.xx; m6[tri(1, 0)] += bI.xy; m6[tri(1, 1)] += bI.yy;
      m6[tri(2, 0)] += bI.xz; m6[tri(2, 1)] += bI.yz; m6[tri(2, 2)] += bI.zz;
      m6[tri(3, 0)] += bx.a00; m6[tri(3, 1)] += bx.a10; m6[tri(3, 2)] += bx.a20;
      m6[tri(4, 0)] += bx.a01; m6[tri(4, 1)] += bx.a11; m6[tri(4, 2)] += bx.a21;
      m6[tri(5, 0)] += bx.a02; m6[tri(5, 1)] += bx.a12; m6[tri(5, 2)] += bx.a22;
      m6[tri(3, 3)] += bm; m6[tri(4, 4)] += bm; m6[tri(5, 5)] += bm;
#pragma unroll
      for (int t = 0; t < 6; t++) z0[t] += envtab[envslot::bias + t];
    }
    float a0[6];
    {
      const Chol6 ch = chol6(m6);
      float bneg[6];
#pragma unroll
      for (int t = 0; t < 6; t++) bneg[t] = -z0[t];
      chol6_solve(ch, bneg, a0);                // acceleration relative to free fall (gravity as a fictitious base acceleration)
      if (l16 == 0) {                           // the factor is needed again by the row images and the final back substitution
#pragma unroll
        for (int t = 0; t < 21; t++) envtab[envslot::chol + t] = ch.l[t];
      }
    }
    // ---------------- joint accelerations of this lane's leg, velocity prediction v* = clamp(v + a dt)
    {
      float t3[3];
#pragma unroll
      for (int m = 0; m < 3; m++) t3[m] = (u[m] - dot6(W[m], a0)) * di[m];
      // qdd = L^-T t3
      const float a2 = t3[2], a1 = fmaf(-L21, a2, t3[1]), a0j = fmaf(-L10, a1, fmaf(-L20, a2, t3[0]));
      const float qdd[3] = {a0j, a1, a2};
      const V3 wd = mul(R, V3{a0[0], a0[1], a0[2]});
      V3 vd = mul(R, V3{a0[3], a0[4], a0[5]} + cross(wb, vb));
      vd.z += P.gz;
      ww = V3{clampf(fmaf(wd.x, dt, ww.x), -P.vmax, P.vmax), clampf(fmaf(wd.y, dt, ww.y), -P.vmax, P.vmax), clampf(fmaf(wd.z, dt, ww.z), -P.vmax, P.vmax)};
      vw = V3{clampf(fmaf(vd.x, dt, vw.x), -P.vmax, P.vmax), clampf(fmaf(vd.y, dt, vw.y), -P.vmax, P.vmax), clampf(fmaf(vd.z, dt, vw.z), -P.vmax, P.vmax)};
#pragma unroll
      for (int t = 0; t < 3; t++) qd[t] = clampf(fmaf(qdd[t], dt, qd[t]), -P.vmax, P.vmax);
    }
    wbs = tmul(R, ww); vbs = tmul(R, vw);
    __syncwarp();                                     // every lane has read F / H: the leg table becomes the rows' table
    if (l16 == 0) {                                   // predicted base velocity for the rows' right-hand sides (any lane of the warp may build them)
      float* v = envtab + envslot::vel;
      v[0] = wbs.x; v[1] = wbs.y; v[2] = wbs.z; v[3] = vbs.x; v[4] = vbs.y; v[5] = vbs.z;
    }
    if (i == 0) {
      float* lt = legtab + k * kLegW;
#pragma unroll
      for (int m = 0; m < 3; m++)
#pragma unroll
        for (int t = 0; t < 6; t++) lt[legrow::W + 6 * m + t] = W[m][t];
      lt[legrow::L] = L10; lt[legrow::L + 1] = L20; lt[legrow::L + 2] = L21;
      lt[legrow::dinv] = di[0]; lt[legrow::dinv + 1] = di[1]; lt[legrow::dinv + 2] = di[2];
      lt[legrow::qd] = qd[0]; lt[legrow::qd + 1] = qd[1]; lt[legrow::qd + 2] = qd[2];
      lt[legrow::c3] = c3; lt[legrow::s3] = s3;       // for the fp64 clearance of the shank's spheres
    }
    }   // ================ end of the forward dynamics
    T16_MARK(1);
    __syncwarp();
    const M3 R = qmat(qp);                            // world <- B' (recomputed: cheaper than keeping nine registers alive)
    // ---------------- PMC hurdle plate: getContactPoints (PLE:343) reports the manifolds built on the last sub-step's pre-step poses
    if (ENV == kPmc && P.has_ob && sub == P.substeps - 1) {
      const int o0 = mc.ob_off[clip], n_ob = mc.ob_off[clip + 1] - o0;
      if (n_ob > 0) {
        const float* lk = linktab + 3 * k * kLinkW;     // links 0, 1, 2 of the leg
        const float c1 = lk[linkrec::c1], s1 = lk[linkrec::s1], c2 = lk[kLinkW + linkrec::cy], s2 = lk[kLinkW + linkrec::sy];
        const float c23 = lk[2 * kLinkW + linkrec::cy], s23 = lk[2 * kLinkW + linkrec::sy];
        const V3 p1 = ld3(lk + linkrec::p), p2 = ld3(lk + kLinkW + linkrec::p), p3 = ld3(lk + 2 * kLinkW + linkrec::p);
        const V3 fb = p3 + rot<0>(rot<1>(ld3(L.foot), c23, s23), c1, s1);     // foot centre of this lane's leg
        const double* ob = mc.ob_table + (size_t)(o0 + ob_id) * 4;
        float sy_, cy_;
        llq_sincosf((float)ob[3], &sy_, &cy_);
        const V3 org = V3{(float)(px - ob[1]), (float)(py - ob[2]), (float)pz};      // base position relative to the plate centre
        const V3 wh = p2 + rot<0>(rot<1>(ld3(M.wheel_off[k]), c2, s2), c1, s1);
        bool hit = plate_hit(org + mul(R, fb), L.foot_r, cy_, sy_, P.ob_hx, P.ob_hy, P.ob_hz, P.breaking);
        hit = hit || plate_hit(org + mul(R, wh), M.wheel_r[k], cy_, sy_, P.ob_hx, P.ob_hy, P.ob_hz, P.breaking);
        hit = hit || plate_hit(org + mul(R, p1), M.hip_r[k], cy_, sy_, P.ob_hx, P.ob_hy, P.ob_hz, P.breaking);
        hit = hit || plate_hit(org + mul(R, ld3(M.corner[2 * k])), 0.f, cy_, sy_, P.ob_hx, P.ob_hy, P.ob_hz, P.breaking);
        hit = hit || plate_hit(org + mul(R, ld3(M.corner[2 * k + 1])), 0.f, cy_, sy_, P.ob_hx, P.ob_hy, P.ob_hz, P.breaking);
        ob_hit = hit;
      }
    }
    // ---------------- SEPMC: getContactPoints() (CTG:426-456) = manifolds of the last sub-step, built on its pre-step poses
    if (ENV == kSepmc && sub == P.substeps - 1) {
      float* srow = &s_new[el][0];
      const float* prow = &s_new[el ^ 1][0];
      const V3 pw = V3{(float)px, (float)py, (float)pz};
      const float* lk = linktab + 3 * k * kLinkW;       // links 0, 1, 2 of the leg
      const float c1 = lk[linkrec::c1], s1 = lk[linkrec::s1], c2 = lk[kLinkW + linkrec::cy], s2 = lk[kLinkW + linkrec::sy];
      const float c23 = lk[2 * kLinkW + linkrec::cy], s23 = lk[2 * kLinkW + linkrec::sy];
      const V3 p1 = ld3(lk + linkrec::p), p2 = ld3(lk + kLinkW + linkrec::p), p3 = ld3(lk + 2 * kLinkW + linkrec::p);
      const V3 fb = p3 + rot<0>(rot<1>(ld3(L.foot), c23, s23), c1, s1);       // foot centre of this lane's leg
      const V3 wh = pw + mul(R, p2 + rot<0>(rot<1>(ld3(M.wheel_off[k]), c2, s2), c1, s1));
      const V3 hp_ = pw + mul(R, p1), ft = pw + mul(R, fb);
      const V3 c0 = pw + mul(R, ld3(M.corner[2 * k])), c1_ = pw + mul(R, ld3(M.corner[2 * k + 1]));
      if (i == 0) {
        float* o = srow + kProxyW * k;
        o[0] = ft.x; o[1] = ft.y; o[2] = ft.z; o[3] = wh.x; o[4] = wh.y; o[5] = wh.z; o[6] = hp_.x; o[7] = hp_.y; o[8] = hp_.z;
        o[9] = c0.x; o[10] = c0.y; o[11] = c0.z; o[12] = c1_.x; o[13] = c1_.y; o[14] = c1_.z;
        if (k < 2) { const V3 hd = pw + mul(R, V3{M.handle[k][0], M.handle[k][1], M.handle[k][2]}); o[15] = hd.x; o[16] = hd.y; o[17] = hd.z; }
      }
      __syncwarp();
      const float fx = (float)PS.flag_x, fy = (float)PS.flag_y;
      // the robot's "body" links (legs + wheels, CTG:427) are represented by its hip and wheel spheres
      bool tch = flag_dist(hp_, fx, fy) - M.hip_r[k] < P.breaking || flag_dist(wh, fx, fy) - M.wheel_r[k] < P.breaking;
      bool tg = false;
#pragma unroll 1
      for (int j = 0; j < 4; j++) {
        const float* pj = prow + kProxyW * j;
        const float rj[6] = {M.leg[j].foot_r, M.wheel_r[j], M.hip_r[j], 0.f, 0.f, M.handle[j & 1][3]};
#pragma unroll
        for (int t = 0; t < 6; t++) {
          if (t == 5 && j >= 2) continue;
          const V3 c = V3{pj[3 * t], pj[3 * t + 1], pj[3 * t + 2]};
          tg = tg || norm3(hp_ - c) - M.hip_r[k] - rj[t] < P.breaking || norm3(wh - c) - M.wheel_r[k] - rj[t] < P.breaking;
        }
      }
      int bits = (tch ? 1 : 0) | (tg ? 2 : 0);
      bits |= __shfl_xor_sync(FULL, bits, 1);
      bits |= __shfl_xor_sync(FULL, bits, 2);
      const int other = __shfl_xor_sync(FULL, bits, 16);
      touch_own = (bits & 1) != 0;
      tag = ((robot == 0 ? bits : other) & 2) != 0;               // only robot 0's body counts (CTG:464)
      __syncwarp();
    }
    __syncwarp();
    // ---------------- collision detection on the pre-step pose: spheres l16 and l16 + 16 against the statics
    const V3 nb = V3{R.a20, R.a21, R.a22};               // world z in base coords
    int nc = 0;
    int mycon[2] = {-1, -1};
    {
      const double qx = qp.x, qy = qp.y, qz = qp.z, qw = qp.w;
      const double nx = 2.0 * (qx * qz - qy * qw), ny = 2.0 * (qy * qz + qx * qw), nz = 1.0 - 2.0 * (qx * qx + qy * qy);
#pragma unroll
      for (int rd = 0; rd < 2; rd++) {
        if (rd * 16 >= nsph) break;                      // warp-uniform
        const int s = rd * 16 + l16;
        const bool have = s < nsph;
        const SphConst& sp = ST.s[have ? s : 0];
        const int sleg = sp.leg, sdep = sp.depth;
        float lc1 = 1.f, ls1 = 0.f, lcy = 1.f, lsy = 0.f;
        V3 lp = V3{0.f, 0.f, 0.f};
        if (sdep > 0) {
          const float* lk = linktab + (3 * sleg + sdep - 1) * kLinkW;
          const float4 a = ld4(lk + linkrec::c1), b4 = ld4(lk + linkrec::p);
          lc1 = a.x; ls1 = a.y; lcy = a.z; lsy = a.w; lp = V3{b4.x, b4.y, b4.z};
        }
        const V3 cl = ld3(sp.c);
        const V3 cb = rotxy(cl, lcy, lsy, lc1, ls1) + lp;          // sphere centre, base coordinates
        float dist = (float)pz + dot(nb, cb) - sp.r;                // fp32 screen
        const bool statics = rule == 2 || s < 4;                    // legacy rules: only the feet touch walls and boxes
        bool near_ = have && dist < P.breaking + 0.01f;
        if (ENV == kSepmc && statics && have) {
          const V3 cw = V3{(float)px, (float)py, (float)pz} + mul(R, cb);
          near_ = near_ || fmaxf(fabsf(cw.x), fabsf(cw.y)) + sp.r > kWallIn - P.breaking - 0.01f;
        }
        unsigned cmask = 0;                              // EPMC corridor: candidate boxes this sphere can touch (fp32 screen, 3 cm of slack)
        if (ENV == kEpmcCorridor && statics && have && n_cand > 0) {
          const V3 cw = V3{(float)px, (float)py, (float)pz} + mul(R, cb);
          const float reach = sp.r + P.aux_r + P.breaking + 0.03f;
          for (int c = 0; c < n_cand; c++) {
            const float* bx = s_cand + 6 * c;
            const float ex = fabsf(cw.x - bx[0]) - bx[3], ey = fabsf(cw.y - bx[1]) - bx[4], ez = fabsf(cw.z - bx[2]) - bx[5];
            if (fmaxf(ex, fmaxf(ey, ez)) < reach) cmask |= 1u << c;
          }
          near_ = near_ || cmask != 0;
        }
        int plane = 0;                                   // 0 ground, 1..4 arena walls (normals -x, +x, -y, +y), 5 a corridor box
        V3 nworld = V3{0.f, 0.f, 1.f};
        if (__any_sync(FULL, near_)) {
          if (near_) {
            // The clearance feeds Bullet's speculative-contact target (-penetration/dt): a 1e-7 m rounding error becomes 5e-5 m/s.
            // Evaluate the sphere centre in fp64 from the fp32 joint sines / cosines (the chain of the link's joints, in double).
            double x = cl.x, y = cl.y, z = cl.z, t;
            if (sdep > 0) {
              const LegConst& SL = M.leg[sleg];
              if (sdep == 3) {
                const double dc3 = (double)legtab[sleg * kLegW + legrow::c3], ds3 = (double)legtab[sleg * kLegW + legrow::s3];
                t = dc3 * x + ds3 * z; z = -ds3 * x + dc3 * z; x = t;            // Ry(theta3)
                x += (double)SL.j[2].r[0]; y += (double)SL.j[2].r[1]; z += (double)SL.j[2].r[2];
              }
              if (sdep >= 2) {
                const float* l1 = linktab + (3 * sleg + 1) * kLinkW;
                const double dc2 = (double)l1[linkrec::cy], ds2 = (double)l1[linkrec::sy];
                t = dc2 * x + ds2 * z; z = -ds2 * x + dc2 * z; x = t;            // Ry(theta2)
                x += (double)SL.j[1].r[0]; y += (double)SL.j[1].r[1]; z += (double)SL.j[1].r[2];
              }
              const double dc1 = lc1, ds1 = ls1;
              t = dc1 * y - ds1 * z; z = ds1 * y + dc1 * z; y = t;               // Rx(q1)
              x += (double)SL.j[0].r[0]; y += (double)SL.j[0].r[1]; z += (double)SL.j[0].r[2];
            }
            dist = (float)(pz + nx * x + ny * y + nz * z - (double)sp.r);
            if ((ENV == kSepmc || ENV == kEpmcCorridor) && statics) {
              const double wx = px + (1.0 - 2.0 * (qy * qy + qz * qz)) * x + 2.0 * (qx * qy - qz * qw) * y + 2.0 * (qx * qz + qy * qw) * z;
              const double wy = py + 2.0 * (qx * qy + qz * qw) * x + (1.0 - 2.0 * (qx * qx + qz * qz)) * y + 2.0 * (qy * qz - qx * qw) * z;
              if (ENV == kSepmc) {
                // the arena walls (BSG:863-902) as four more half-spaces; one contact per sphere, the deepest (DESIGN.md 5)
                const double lim = (double)kWallIn - (double)sp.r;
                const float d1 = (float)(lim - wx), d2 = (float)(lim + wx), d3 = (float)(lim - wy), d4 = (float)(lim + wy);
                if (d1 < dist) { dist = d1; plane = 1; }
                if (d2 < dist) { dist = d2; plane = 2; }
                if (d3 < dist) { dist = d3; plane = 3; }
                if (d4 < dist) { dist = d4; plane = 4; }
              } else {
                // EPMC corridor: sphere vs the candidate boxes, in fp64 like the ground clearance; one contact per sphere, the deepest
                const double wz = pz + nx * x + ny * y + nz * z;
                for (unsigned cm = cmask; cm; cm &= cm - 1) {
                  const int c = __ffs((int)cm) - 1;
                  double db; V3 nn;
                  const float* bx = s_cand + 6 * c;
                  sphere_box(wx, wy, wz, (double)sp.r, bx, db, nn);
                  if ((float)db < dist) { dist = (float)db; plane = 5; nworld = nn; }
                  // the element's two auxiliary cylinders (BSE:43-104): along y on the box's x faces, on its top edge (bars: bottom edge);
                  // the 200 m walls carry none
                  if (P.aux_r > 0.f && bx[3] < 50.f && fabs(wy - (double)bx[1]) <= (double)bx[4]) {
                    const double ez = (double)bx[2] + (P.element_id == 2 ? -(double)bx[5] : (double)bx[5]), dz = wz - ez;
#pragma unroll
                    for (int side = -1; side <= 1; side += 2) {
                      const double dx = wx - ((double)bx[0] + (double)side * (double)bx[3]), len = sqrt(dx * dx + dz * dz);
                      const double dc = len - (double)P.aux_r - (double)sp.r;
                      if (len > 0.0 && (float)dc < dist) { dist = (float)dc; plane = 5; nworld = V3{(float)(dx / len), 0.f, (float)(dz / len)}; }
                    }
                  }
                }
              }
            }
          }
        }
        bool contact = have && dist < P.breaking;
        if (rule == 1 && rd == 0) {
          // legacy rule (llq_config.knee_contacts = 1): one contact per leg, the deeper of {foot, knee wheel}; the foot wins ties
          const float od = __shfl_xor_sync(FULL, dist, 4);
          const bool oc = __shfl_xor_sync(FULL, contact ? 1 : 0, 4) != 0;
          if (l16 < 4) contact = contact && !(oc && od < dist);
          else if (l16 < 8) contact = contact && !(oc && od <= dist);
        }
        const unsigned bal = (__ballot_sync(FULL, contact) >> (tid & 16)) & 0xFFFFu;
        int idx = nc + __popc(bal & ((1u << l16) - 1u));    // manifold points in sphere order
        if (rule == 1) idx = __popc((bal | (bal >> 4)) & ((1u << (l16 & 3)) - 1u));   // legacy rule: in leg order (one point per leg)
        nc += __popc(bal);
        if (contact && idx >= kMaxCon) { contact = false; n_overflow += 1; }
        if (contact) {
          // directions (base coordinates): normal, then btPlaneSpace1's two tangents
          V3 dn = nb, d1_ = neg(V3{R.a10, R.a11, R.a12}), d2_ = V3{R.a00, R.a01, R.a02};   // ground: n = +z, t1 = -y, t2 = +x (world)
          if (ENV == kSepmc && plane != 0) {
            const V3 w0 = V3{R.a00, R.a01, R.a02}, w1 = V3{R.a10, R.a11, R.a12};
            d2_ = nb;                                     // t2 = +z for every wall
            if (plane == 1) { dn = neg(w0); d1_ = neg(w1); }
            else if (plane == 2) { dn = w0; d1_ = w1; }
            else if (plane == 3) { dn = neg(w1); d1_ = w0; }
            else { dn = w1; d1_ = neg(w0); }
          }
          if (ENV == kEpmcCorridor && plane == 5) {                   // general normal: btPlaneSpace1 in world axes, then into base coordinates
            const V3 n = nworld;
            V3 t1, t2;
            if (fabsf(n.z) > 0.70710678118654752f) {
              const float a = n.y * n.y + n.z * n.z, kk = rsqrtf(a);
              t1 = V3{0.f, -n.z * kk, n.y * kk};
              t2 = V3{a * kk, -n.x * t1.z, n.x * t1.y};
            } else {
              const float a = n.x * n.x + n.y * n.y, kk = rsqrtf(a);
              t1 = V3{-n.y * kk, n.x * kk, 0.f};
              t2 = V3{-n.z * t1.y, n.z * t1.x, a * kk};
            }
            dn = tmul(R, n); d1_ = tmul(R, t1); d2_ = tmul(R, t2);
          }
          const V3 Pc = cb - sp.r * dn;                   // contact point on the sphere surface
          float* cr = contab + idx * kConW + conrec::leg;
          st4(cr, __int_as_float(sdep > 0 ? sleg : -1), __int_as_float(sdep), Pc.x, Pc.y);
          st4(cr + 4, Pc.z, dn.x, dn.y, dn.z);
          st4(cr + 8, d1_.x, d1_.y, d1_.z, d2_.x);
          st4(cr + 12, d2_.y, d2_.z, dist, sp.foot ? mu_foot : sp.mu_link);
          cr[conrec::lam0] = P.warm * warm[rd]; cr[conrec::lam] = 0.f;
          mycon[rd] = idx;
        } else {
          warm[rd] = 0.f;                                 // manifold point removed: no warm start
        }
      }
      if (nc > kMaxCon) nc = kMaxCon;
    }
    // ---------------- joint-limit rows (btMultiBodyJointLimitConstraint: a row exists only while the limit is violated)
    int nl = 0;
    {
      float dir = 0.f, pen = 0.f;
      const int ic = i < 3 ? i : 0;
      if (i < 3 && L.j[ic].haslim) {
        const float qi = i == 0 ? q[0] : (i == 1 ? q[1] : q[2]);
        if (qi - L.j[ic].lower <= 0.f) { dir = 1.f; pen = qi - L.j[ic].lower; }
        else if (L.j[ic].upper - qi <= 0.f) { dir = -1.f; pen = L.j[ic].upper - qi; }
      }
      const unsigned bal = (__ballot_sync(FULL, dir != 0.f) >> (tid & 16)) & 0xFFFFu;
      nl = __popc(bal);
      const int rk = __popc(bal & lowmask);
      if (dir != 0.f) {
        if (rk < kMaxLim) st4(limtab + rk * kLimW + limrec::leg, __int_as_float(k), __int_as_float(i), dir, pen);
        else n_overflow += 1;
      }
      if (nl > kMaxLim) nl = kMaxLim;
    }
    __syncwarp();
    T16_MARK(2);
    float dvb[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, dvl[3] = {0.f, 0.f, 0.f};
    // ---------------- the rows of the CTA's envs: publish the counts, pair the envs by load, solve, hand the totals back
    if (l16 == 0) s_cnt[el] = nc | (nl << 8);
    __syncthreads();           // every env's tables (links, legs, contacts, limits, Cholesky factor, predicted velocity) are complete
    T16_MARK(0);
    {
      // Pairing: the critical path of the sub-step is the longest row list of the CTA (the sweep is sequential within an env), and a
      // warp whose two envs have more than 32 rows between them needs two passes -- so warp w takes the env of rank w (by row count,
      // descending) together with the env of rank EPB - 1 - w.  The result does not depend on the pairing (an env's rows only meet
      // its own tables).
      const int lane = tid & 31, wq = tid >> 5;
      const int cnt = lane < EPB ? s_cnt[lane] : 0;
      const int nrow = 3 * (cnt & 255) + (cnt >> 8);
      int rank = 0;
#pragma unroll 1
      for (int j = 0; j < EPB; j++) {
        const int nj = __shfl_sync(FULL, nrow, j);
        rank += (nj > nrow || (nj == nrow && j < lane)) ? 1 : 0;
      }
      const int ea = __ffs(__ballot_sync(FULL, lane < EPB && rank == wq)) - 1;
      const int eb = __ffs(__ballot_sync(FULL, lane < EPB && rank == EPB - 1 - wq)) - 1;
      const int ca_ = __shfl_sync(FULL, cnt, ea), cb_ = __shfl_sync(FULL, cnt, eb);
      // (redux results live in uniform registers: the guards below compile to uniform branches)
      const int cA = __reduce_max_sync(FULL, ca_ & 255), lA = __reduce_max_sync(FULL, ca_ >> 8);
      const int cB = __reduce_max_sync(FULL, cb_ & 255), lB = __reduce_max_sync(FULL, cb_ >> 8);
      const int eA = __reduce_max_sync(FULL, ea), eB = __reduce_max_sync(FULL, eb);
      const int nA = 3 * cA + lA, nB = 3 * cB + lB;
      T16_ADD(6, max(cA, cB) * 256 + max(lA, lB) + (nA > 16 || nB > 16 ? 65536 : 0) + (nA + nB > 32 ? (1 << 24) : 0));
      if (nA | nB) {
        RowsIn in;
#ifdef LLQ16_TIMING
        in.t16 = t16_; in.t16c = &t16_c;
#endif
        in.lane = lane; in.acol = s_atab + wq * kATabWarp + lane;
        in.dt = dt; in.slop = P.slop; in.erp = P.erp; in.jerp = P.jerp; in.max_imp = P.max_imp; in.iters = P.solver_iters;
        float* const tbA = s_env_dyn + eA * kEnvFloats;
        float* const tbB = s_env_dyn + eB * kEnvFloats;
        const bool two_pass = nA + nB > 32;            // more rows than lanes: env A on all 32 lanes, then env B
#pragma unroll 1
        for (int pass = 0; pass < (two_pass ? 2 : 1); pass++) {
          const int split = two_pass ? (pass == 0 ? 32 : 0) : ((nA <= 16 && nB <= 16) ? 16 : (nA > 16 ? nA : 32 - nB));
          const bool X = lane >= split;
          in.tb = X ? tbB : tbA;
          in.nc = X ? cB : cA; in.nl = X ? lB : lA;
          in.lane0 = X ? split : 0; in.rr = lane - in.lane0; in.split = split;
          in.Cmax = two_pass ? (pass == 0 ? cA : cB) : max(cA, cB);
          in.Lmax = two_pass ? (pass == 0 ? lA : lB) : max(lA, lB);
          const bool upper = lane >= 16;
          in.res = (two_pass && upper != (pass == 1)) ? nullptr : (upper ? tbB : tbA) + (rowtab - linktab);
          solve_rows(in);
          __syncwarp();
        }
      }
    }
    __syncthreads();           // the totals of every env of the CTA are in its row table
    T16_MARK(3);
    if (nc | nl) {
      if (l16 == 0) { n_contact_rows += 3u * (unsigned)nc; n_limit_rows += (unsigned)nl; }
#pragma unroll
      for (int rd = 0; rd < 2; rd++) if (mycon[rd] >= 0) warm[rd] = contab[mycon[rd] * kConW + conrec::lam];
      // ---- total impulse -> velocity change: one back substitution for the base, one 3x3 solve per leg
      const float* yt = rowtab + sums::base;
      const float4 y0 = ld4(yt), y1 = ld4(yt + 4);
      const float Yt[6] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y};
      const float om[3] = {rowtab[sums::leg + 3 * k], rowtab[sums::leg + 1 + 3 * k], rowtab[sums::leg + 2 + 3 * k]};
      chol6_bwd_p(envtab + envslot::chol, Yt, dvb);
      const float* lt = legtab + k * kLegW;        // W, L, D^-1 of this lane's leg come back from the leg table (not kept live across the solve)
      float t3[3];
#pragma unroll
      for (int m = 0; m < 3; m++) {
        const float wm[6] = {lt[legrow::W + 6 * m], lt[legrow::W + 6 * m + 1], lt[legrow::W + 6 * m + 2], lt[legrow::W + 6 * m + 3],
                             lt[legrow::W + 6 * m + 4], lt[legrow::W + 6 * m + 5]};
        t3[m] = (om[m] - dot6(wm, dvb)) * lt[legrow::dinv + m];
      }
      // L = (L10, L20, L21)
      dvl[2] = t3[2]; dvl[1] = fmaf(-lt[legrow::L + 2], dvl[2], t3[1]); dvl[0] = fmaf(-lt[legrow::L], dvl[1], fmaf(-lt[legrow::L + 1], dvl[2], t3[0]));
    }
    __syncwarp();              // the row table is the next sub-step's scratch
    T16_MARK(3);
    // ---------------- apply the impulses, clamp, integrate (btMultiBody::stepPositionsMultiDof)
    {
      V3 dw = mul(R, V3{dvb[0], dvb[1], dvb[2]}), dv = mul(R, V3{dvb[3], dvb[4], dvb[5]});
      ww = V3{clampf(ww.x + dw.x, -P.vmax, P.vmax), clampf(ww.y + dw.y, -P.vmax, P.vmax), clampf(ww.z + dw.z, -P.vmax, P.vmax)};
      vw = V3{clampf(vw.x + dv.x, -P.vmax, P.vmax), clampf(vw.y + dv.y, -P.vmax, P.vmax), clampf(vw.z + dv.z, -P.vmax, P.vmax)};
#pragma unroll
      for (int t = 0; t < 3; t++) {
        qd[t] = clampf(qd[t] + dvl[t], -P.vmax, P.vmax);
        q[t] = fmaf(qd[t], dt, q[t]);
      }
      px += (double)vw.x * P.sim_dt; py += (double)vw.y * P.sim_dt; pz += (double)vw.z * P.sim_dt;
      float fa = norm3(ww);
      float sc;
      sc = 0.5f * dt - dt * dt * dt * 0.020833333333f * fa * fa;      // used below 1e-3 rad/s (btMultiBody's series)
      float sh, chh;
      llq_sincosf(0.5f * fa * dt, &sh, &chh);
      if (!(fa < 0.001f)) sc = sh / fa;
      Q4 dq = Q4{sc * ww.x, sc * ww.y, sc * ww.z, chh};
      qp = qnormalize(qmul(dq, qp));
    }
    bad = bad || !(fabsf(qd[0]) <= P.vmax) || !(fabsf(ww.x) <= P.vmax) || !(fabsf(vw.x) <= P.vmax);
    // ---------------- mocap clock (PLE:208-210): sampled with the time *before* the increment
    if (ENV == kPmc && sub == P.substeps - 1) {
      frame_id = (int)floor(time / P.frame_dt);
      frame_frac = (time - frame_id * P.frame_dt) / P.frame_dt;
      const int last = mc.clip_off[clip + 1] - mc.clip_off[clip] - P.margin + 2;     // see llq_kernels.cuh: runaway cursors only
      if (frame_id > last) { frame_id = last; frame_frac = 0.0; }
      if (frame_id < 0) { frame_id = 0; frame_frac = 0.0; }
    }
    time += P.sim_dt;
  }
  __syncwarp();

  // ================= end of the policy step: hand the state over to the tail lanes (4 per env, 8 envs per warp) =================
  {
    int bi = bad ? 1 : 0;
    bi |= __shfl_xor_sync(FULL, bi, 1); bi |= __shfl_xor_sync(FULL, bi, 2); bi |= __shfl_xor_sync(FULL, bi, 4); bi |= __shfl_xor_sync(FULL, bi, 8);
    bad = bi != 0;
  }
  if (valid) {                                             // contact memory of this lane's two spheres
    if (l16 < nsph) E.warm[(size_t)l16 * N + env] = warm[0];
    if (16 + l16 < nsph) E.warm[(size_t)(16 + l16) * N + env] = warm[1];
  }
  {
    TailState* T = reinterpret_cast<TailState*>(rowtab);
    if (l16 == 0) {
      T->px = px; T->py = py; T->pz = pz; T->time = time; T->frame_frac = frame_frac;
      T->frame_id = frame_id; T->ob_id = ob_id; T->push_count = push_count; T->push_draws = push_draws;
      T->pf[0] = pf[0]; T->pf[1] = pf[1]; T->pf[2] = pf[2];
      T->qp[0] = qp.x; T->qp[1] = qp.y; T->qp[2] = qp.z; T->qp[3] = qp.w;
      T->vw[0] = vw.x; T->vw[1] = vw.y; T->vw[2] = vw.z; T->ww[0] = ww.x; T->ww[1] = ww.y; T->ww[2] = ww.z;
    }
    // ob_hit / touch / tag are per-leg partial results: fold them over the legs here
    int fl = (bad ? tflag::bad : 0) | (ob_hit ? tflag::ob_hit : 0) | (touch_own ? tflag::touch_own : 0) | (tag ? tflag::tag : 0);
    fl |= __shfl_xor_sync(FULL, fl, 1); fl |= __shfl_xor_sync(FULL, fl, 2);
    if (l16 == 0) T->flags = fl;
    if (i == 0) {
#pragma unroll
      for (int t = 0; t < 3; t++) { T->q[3 * k + t] = q[t]; T->qd[3 * k + t] = qd[t]; }
    }
  }
  // counters: one atomic per warp
  {
    unsigned cr = n_contact_rows, lr = n_limit_rows, ov = n_overflow;
    if (!valid) { cr = 0; lr = 0; ov = 0; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { cr += __shfl_xor_sync(FULL, cr, o); lr += __shfl_xor_sync(FULL, lr, o); ov += __shfl_xor_sync(FULL, ov, o); }
    if ((threadIdx.x & 31) == 0) {
      if (cr) atomicAdd(&E.counters[2], (unsigned long long)cr);
      if (lr) atomicAdd(&E.counters[3], (unsigned long long)lr);
      if (ov) atomicAdd(&E.counters[5], (unsigned long long)ov);
    }
  }
  __pipeline_wait_prior(0);                                // this thread's share of the history prefetch has landed
  __syncthreads();
  if (tid < 4 * EPT) {
    const int tel = tid >> 2, tk = tid & 3;
    const bool tval = tel < EPB && blockIdx.x * EPB + tel < N;          // surplus lanes shadow the CTA's last env into a dummy staging row
    const int tsrc = tel < EPB ? tel : EPB - 1;
    const int tenv_raw = blockIdx.x * EPB + tsrc;
    const float* tbase = s_env_dyn + tsrc * kEnvFloats;
    step_tail<ENV>(E, mc, P, M, &s_new[0][0], &s_hist[0][0], *reinterpret_cast<const TailState*>(tbase + (rowtab - linktab)),
                        tbase + (envtab - linktab) + envslot::act, obs2, obs2_ld, winner, seed, gid0, record, tel, tk, tenv_raw < N ? tenv_raw : N - 1, tval);
  }
  // ---- observation rows (history shift + new prop / action / future; EPMC / SEPMC: the 778 perception rays are cast while the row is
  // written): every warp of the CTA emits the rows of its own two envs, coalesced
  __syncthreads();
  emit_obs_rows<ENV, 2>(E.obs, obs2, obs2_ld, &s_new[(tid >> 5) << 1][0], &s_hist[(tid >> 5) << 1][0], warp_env0, N, 0, 0x3u, E.boxes);
#ifdef LLQ16_TIMING
  T16_MARK(4);
  t16_[7] = clock64() - t16_s;
  if ((tid & 31) == 0) {
    const int gw = blockIdx.x * (BLOCK / 32) + (tid >> 5);
    if (gw < 16384) for (int t = 0; t < 12; t++) g_t16[gw * 12 + t] = (unsigned long long)t16_[t];
  }
#endif
}

}  // namespace llq
