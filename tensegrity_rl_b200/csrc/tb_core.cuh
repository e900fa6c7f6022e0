// tb_core.cuh -- bar-lane tensegrity physics for sm_100a: THREE LANES PER ENV (one per bar), TEN ENVS PER WARP.
//
// What is computed is MuJoCo 2.3.7's mj_forward / mj_step for the 3-bar model (SURVEY.md App. B; the reference reaches
// it through gym's MujocoEnv.do_simulation, tr_env.py:346,812, tensegrity_env.py:297): free-joint kinematics ->
// 9 two-site spatial tendons -> collision (plane / height field / bar-bar, MPR where MuJoCo uses libccd) -> condim-6
// elliptic contact rows -> Newton with exact line search -> implicitfast -> advance.
//
// Mapping.  A bar's pose / velocity / acceleration and every per-bar vector of the solver live in the REGISTERS of the
// bar's lane for all frame_skip substeps.  Everything that crosses bars lives in the env's slice of SHARED memory:
// world-frame poses and twists, the contacts (a small pool of slots per env; slots beyond it spill to a per-env global
// area), and the 6x6 blocks of the Newton Hessian.  There are no per-lane local arrays on the hot path: local memory is
// interleaved across the 32 lanes of a warp, so an array only one lane of an env uses still costs 32 lanes of cache.
// Work that is naturally per contact is done by the lane that found the contact (its owner); work that is per bar
// (wrench gathering, diagonal Hessian blocks, the bar's block row of the factorisation) by the bar's lane, so a
// bar-bar contact is processed by up to three lanes in parallel.  Control flow is UNIFORM across the warp (in the step
// kernel at some loop heads across the CTA: uni_any): every data-dependent loop (Newton iterations, line-search
// evaluations, second forward pass after a bad acceleration) runs while ANY env needs it, the others predicated off, so
// the envs of a warp share every fetched instruction and never need a partial barrier.
#pragma once
#include "tb_mpr.h"

namespace tb {

constexpr int G = 3;        // lanes per env
constexpr int EPW = 10;     // envs per warp (lanes 30, 31 idle)
constexpr int KP = 1;       // contacts per lane held in shared memory; a lane's later contacts live in its part of the
constexpr int KS = 16;      // env's global spill area (KS slots per lane).  Slot addresses depend on (lane, k) only, so
constexpr int NCS = 3 * KP; // the order in which contacts are summed never depends on timing.
constexpr int MAXCL = KP + KS;   // contacts one lane can own (a bar lying flat on the floor: 14)
constexpr int ZONE_TOP = 0, ZONE_BOTTOM = 1, ZONE_MIDDLE = 2;

// Arithmetic of a build.  `real`: kinematics, tendons, collision, integration.  `sreal`: the constraint solver (contact
// rows, Newton Hessian, line search) -- the contact stiffness spans 1e6 x the bar inertia, so the solve needs fp64 to
// stay within 1e-4 of the reference (pure fp32 lands at 1e-3 .. 1e-2: measured with the emulator, DESIGN.md).
struct P64 { typedef double real; typedef double sreal; static constexpr bool per_env = false; };
struct P32 { typedef float real; typedef double sreal; static constexpr bool per_env = false; };   // the optional fp32 mode: fp32 geometry, fp64 solver
// The per-env-parameter variant of a build: the tendon and actuator constants come from the env's row of per-env
// parameters in global memory (NPARAM doubles, PRM_* in tb_model.h) instead of the model.  A separate instantiation,
// so that the kernels of handles without per-env parameters stay exactly what they are.
template <typename B> struct PerEnv : B { static constexpr bool per_env = true; };

// one contact.  Written by its owner lane; read by the lanes of the bars it touches.
template <typename real>
struct Con {
  real frame[9];
  real r1[3], r2[3];   // contact point relative to the centre of body 1 / body 2 (world axes)
  real jar[6], jv[6];
  real wr[6];          // world-frame wrench (force, torque) of the current contact force
  real D0;
  union {
    struct { real bw[6], wcoef, ca, cb; } h;                     // cone state for the Hessian, world frame (eval -> assembly)
    struct { real U0, V0, UU, UV, VV, q0, q1, q2; } ls;          // line-search coefficients (line search only)
  } t;
  int b1, b2;          // bar index 0..2, or -1 for the world (b1 only)
  int zone, owner;     // owner: lane (bar index) that processes the contact, -1 = empty slot
};

// per-env slice of shared memory; the per-env variant also holds the address of the env's parameter row
template <bool PE> struct EnvShRow {};
template <> struct EnvShRow<true> { const double* prm; };
template <typename P>
struct EnvSh : EnvShRow<P::per_env> {
  typedef typename P::real real;
  typedef typename P::sreal sreal;
  // world-frame exchange, rewritten by every pass; xpos / xmat / sph / tlen double as the "stale" kinematics the
  // reference's observation reads (positions lag qpos by one substep)
  real xpos[9], xmat[27], sph[18], tlen[NTEN];
  union {
    struct { real vw[18], actdot[NACT]; };   // world-frame velocities, activation derivatives (within a pass)
    real cfrc[24];                           // mj_rnePostConstraint of the last pass
  };
  double ctrl[NACT], act[NACT];
  union {
    struct { double qpos[NQ], qvel[NV], warm[NV]; } home;   // env state between physics calls (HBM record precision)
    real site[NEND * 3];                                    // tendon end points (tendon stage)
    struct {                                                // Newton solver
      sreal D[3][21];     // diagonal blocks, packed lower; after factorisation unit L below the diagonal, d on it
      sreal O[3][36];     // blocks below the diagonal, full 6x6 row-major: pairs (1,0), (2,0), (2,1)
      sreal dinv[NV];
      sreal xv[NV];       // world-frame twists of the vector under J; during the solve: the block rows' partial solutions
    } sol;
  } u;
  Con<sreal> con[NCS];
  Con<sreal>* spill;      // global memory: 3 * KS slots of this env-in-flight
  int ncl[3];             // contacts owned by each lane
  int ngl[3];             // ... of which the first ngl are ground contacts (world - own bar); bar-bar contacts follow
  int cpl[3];             // which blocks below the diagonal exist (set by the pair owners)
  int nact, overflow, bad, niter, nls, nmpr;
  sreal barforce;
  double action[NACT];    // env layer (lane 0 of the env)
};

struct LaneCtx { int lane, grp, bar, base; bool valid; };
// epw <= EPW: envs this warp works on (its remaining lanes idle along, aliasing the last env's slice read-only)
TB_FN LaneCtx make_lane(int epw = EPW) {
  LaneCtx L;
  L.lane = simt_lane();
  L.valid = L.lane < G * epw;
  L.grp = L.valid ? L.lane / G : epw - 1;
  L.bar = L.lane % G;
  L.base = L.grp * G;
  return L;
}
template <typename real> TB_FN real sum3(real v, int base) {
  real a = shfl(v, base), b = shfl(v, base + 1), c = shfl(v, base + 2);
  return (a + b) + c;
}
TB_FN int isum3(int v, int base) { return shfl(v, base) + shfl(v, base + 1) + shfl(v, base + 2); }
TB_FN bool grp_any(bool p, int base) { return ((ballot(p) >> base) & 7u) != 0; }
// loop conditions: uniform over the warp, or over the CTA when its warps run aligned (they then share fetched
// instructions).  Aligned, this is a CTA barrier, so every warp of the CTA must execute the same sequence of these
// calls: one at every substep (simulate()), and in phys() at the top of every Newton iteration and at mj_checkAcc.
TB_FN bool uni_any(bool p, bool aligned) {
#if TB_DEV
  if (aligned) return __syncthreads_or(p ? 1 : 0) != 0;
#endif
  (void)aligned;
  return any(p);
}

template <typename P> struct BarState { typename P::real x[3], q[4], v[6]; typename P::sreal warm[6]; };

// k-th contact of lane `owner`
template <typename P> TB_FN Con<typename P::sreal>& con_of(EnvSh<P>& S, int owner, int k) {
  if (k < KP) return S.con[owner * KP + k];
  return S.spill[owner * KS + k - KP];
}

// ------------------------------------------------------------------ contact helpers
template <typename real> TB_FN void make_frame(real* f) {
  normalize3(f);
  f[3] = f[4] = f[5] = 0;
  if (f[1] < real(0.5) && f[1] > real(-0.5)) f[4] = 1; else f[5] = 1;
  real t = dot3(f, f + 3);
  addscl3(f + 3, f, -t);
  normalize3(f + 3);
  cross3(f + 6, f, f + 3);
}
// out = J x, x given as world-frame twists per bar (lin, world angular) in xv
template <typename real, typename V> TB_FN void con_mulJ(const Con<real>& c, const V* xvv, real* out) {
  real v2[6], rel[3], relw[3], t[3];   // statically indexed copies only: a dynamically indexed array would live in local memory
  const V* p2 = xvv + 6 * c.b2;
  for (int k = 0; k < 6; k++) v2[k] = (real)p2[k];
  cross3(t, v2 + 3, c.r2);
  add3(rel, v2, t);
  copy3(relw, v2 + 3);
  if (c.b1 >= 0) {
    real v1[6], u1[3];
    const V* p1 = xvv + 6 * c.b1;
    for (int k = 0; k < 6; k++) v1[k] = (real)p1[k];
    cross3(t, v1 + 3, c.r1);
    add3(u1, v1, t);
    sub3(rel, rel, u1); sub3(relw, relw, v1 + 3);
  }
  for (int a = 0; a < 3; a++) { out[a] = dot3(c.frame + 3 * a, rel); out[3 + a] = dot3(c.frame + 3 * a, relw); }
}
template <typename real, typename MR> TB_FN real impedance(const ModelT<MR>& m, real pos) {
  const real MINIMP = real(0.0001), MAXIMP = real(0.9999);
  real d0 = clampr((real)m.solimp[0], MINIMP, MAXIMP), dw = clampr((real)m.solimp[1], MINIMP, MAXIMP);
  real width = tmax(Lim<real>::MINVAL, (real)m.solimp[2]), mid = clampr((real)m.solimp[3], MINIMP, MAXIMP), power = tmax(real(1), (real)m.solimp[4]);
  if (d0 == dw || width <= Lim<real>::MINVAL) return real(0.5) * (d0 + dw);
  real x = tdiv(tabs(pos), width), y;
  if (x >= 1) return dw;
  if (x == 0) return d0;
  if (power == 1) y = x;
  else if (power == 2) y = (x <= mid) ? trcp(mid) * (x * x) : 1 - trcp(1 - mid) * ((1 - x) * (1 - x));
  else if (x <= mid) y = (real)((1 / pow((double)mid, (double)power - 1)) * pow((double)x, (double)power));
  else y = (real)(1 - (1 / pow(1 - (double)mid, (double)power - 1)) * pow(1 - (double)x, (double)power));
  return d0 + y * (dw - d0);
}
// mj_constraintUpdate for one elliptic contact at jar (+ jv if addjv): returns its cost; full: also the contact force
// as a world wrench, the zone and the Hessian weights
template <typename real, typename MR> TB_FN real con_update(Con<real>& c, const ModelT<MR>& m, bool full, bool addjv) {
  real ja[6], U[6], T = 0, mu = (real)m.mu;
  for (int j = 0; j < 6; j++) ja[j] = addjv ? c.jar[j] + c.jv[j] : c.jar[j];
  U[0] = ja[0] * mu;
  for (int j = 1; j < 6; j++) { U[j] = ja[j] * m.fr[j - 1]; T += U[j] * U[j]; }
  real N = U[0], f[6];
  T = tsqrt(T);
  real cost;
  if (N >= mu * T || (T <= 0 && N >= 0)) {
    if (!full) return 0;
    for (int j = 0; j < 6; j++) f[j] = 0;
    c.zone = ZONE_TOP; c.t.h.wcoef = c.t.h.ca = c.t.h.cb = 0;
    cost = 0;
  } else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
    real s = 0;
    for (int j = 0; j < 6; j++) {
      real D = c.D0 * m.dscale[j];
      s += real(0.5) * D * ja[j] * ja[j];
      f[j] = -D * ja[j];
    }
    if (!full) return s;
    c.zone = ZONE_BOTTOM; c.t.h.wcoef = c.D0; c.t.h.ca = c.t.h.cb = 0;
    cost = s;
  } else {
    real Dm = c.D0 * m.inv_mu2, NT = N - mu * T;
    cost = real(0.5) * Dm * NT * NT;
    if (!full) return cost;
    real invT = trcp(T);
    f[0] = -Dm * NT * mu;
    real kap = mu * mu - mu * N * invT;
    real su[6];
    su[0] = 0;
    for (int j = 1; j < 6; j++) {
      f[j] = -f[0] * invT * U[j] * m.fr[j - 1];
      su[j] = m.fr[j - 1] * U[j] * invT;
    }
    // b = sum_j su_j J_j as a world-frame 6-vector (linear part from the tangents, angular part from all three axes)
    for (int k = 0; k < 3; k++) {
      c.t.h.bw[k] = c.frame[3 + k] * su[1] + c.frame[6 + k] * su[2];
      c.t.h.bw[3 + k] = c.frame[k] * su[3] + c.frame[3 + k] * su[4] + c.frame[6 + k] * su[5];
    }
    c.t.h.ca = Dm; c.t.h.cb = Dm * kap; c.t.h.wcoef = c.t.h.cb; c.zone = ZONE_MIDDLE;
  }
  for (int k = 0; k < 3; k++) {
    c.wr[k] = c.frame[k] * f[0] + c.frame[3 + k] * f[1] + c.frame[6 + k] * f[2];
    c.wr[3 + k] = c.frame[k] * f[3] + c.frame[3 + k] * f[4] + c.frame[6 + k] * f[5];
  }
  return cost;
}
// cost and its first two derivatives along the search direction at step a, for one contact
// (coefficients: U0, V0, UU, UV, VV, q0, q1, q2, D0 -- of a contact in memory, or cached in registers by the caller)
template <typename real> struct LsCoef { real U0, V0, UU, UV, VV, q0, q1, q2, D0; };
template <typename real> TB_FN LsCoef<real> ls_coef(const Con<real>& k) {
  LsCoef<real> c;
  c.U0 = k.t.ls.U0; c.V0 = k.t.ls.V0; c.UU = k.t.ls.UU; c.UV = k.t.ls.UV; c.VV = k.t.ls.VV;
  c.q0 = k.t.ls.q0; c.q1 = k.t.ls.q1; c.q2 = k.t.ls.q2; c.D0 = k.D0;
  return c;
}
template <typename real, typename MR> TB_FN void con_ls(const LsCoef<real>& k, const ModelT<MR>& m, real a, real& cost, real& d0, real& d1) {
  real mu = (real)m.mu;
  const real U0 = k.U0, V0 = k.V0, UU = k.UU, UV = k.UV, VV = k.VV;
  real N = U0 + a * V0, Tsqr = UU + a * (2 * UV + a * VV);
  bool bottom = false;
  if (Tsqr <= 0) { if (N < 0) bottom = true; }
  else {
    real T = tsqrt(Tsqr);
    if (N >= mu * T) {}
    else if (mu * N + T <= 0) bottom = true;
    else {
      real invT = trcp(T);
      real N1 = V0, T1 = (UV + a * VV) * invT;
      real T2 = VV * invT - (UV + a * VV) * T1 * (invT * invT);
      real NT = N - mu * T, Dm = k.D0 * m.inv_mu2;
      cost += real(0.5) * Dm * NT * NT;
      d0 += Dm * NT * (N1 - mu * T1);
      d1 += Dm * ((N1 - mu * T1) * (N1 - mu * T1) + NT * (-mu * T2));
    }
  }
  if (bottom) { cost += a * a * k.q2 + a * k.q1 + k.q0; d0 += 2 * a * k.q2 + k.q1; d1 += 2 * k.q2; }
}

// ---- Hessian of one contact in world-frame coordinates (per bar: linear dofs, world angular dofs).
// With J = G T (G: the contact frame applied to the relative twist at the contact point, T = [I, -[r]x ; 0, I] per
// side) a contact contributes T^T K T, K = G^T W G.  Friction is isotropic in the tangent plane (two equal sliding and
// two equal rolling coefficients), so the diagonal part of W gives K = blockdiag(w1 I + (w0 - w1) n n^T,
// w4 I + (w3 - w4) n n^T) in closed form, n = contact normal; a middle-zone cone adds the rank-one terms
// ca a a^T - cb b b^T with b stored in the contact (world frame) and a = mu (n - b_lin, -b_ang).
template <typename real> struct ConW { real wl0, wl1, wa3, wa4; };
template <typename real, typename MR> TB_FN ConW<real> con_weights(const Con<real>& c, const ModelT<MR>& m) {
  const MR* wt = m.wtab[c.zone == ZONE_MIDDLE ? 1 : 0];
  ConW<real> w;
  w.wl0 = c.t.h.wcoef * wt[0]; w.wl1 = c.t.h.wcoef * wt[1]; w.wa3 = c.t.h.wcoef * wt[3]; w.wa4 = c.t.h.wcoef * wt[4];
  return w;
}
// H (packed lower 6x6) += w j j^T
template <typename real> TB_FN void rank1_sym(real* H, real w, const real* j) {
  TB_UNROLL
  for (int i = 0, e = 0; i < 6; i++) {
    real wi = w * j[i];
    TB_UNROLL
    for (int k = 0; k <= i; k++, e++) H[e] += wi * j[k];
  }
}
// X (6x6 row-major) += w a b^T
template <typename real> TB_FN void rank1_gen(real* X, real w, const real* a, const real* b) {
  TB_UNROLL
  for (int i = 0; i < 6; i++) {
    real wi = w * a[i];
    TB_UNROLL
    for (int k = 0; k < 6; k++) X[6 * i + k] += wi * b[k];
  }
}
// cone vectors of a side: u = T^T v = (v_lin, r x v_lin + v_ang) for v = a, b
template <typename real, typename MR> TB_FN void cone_side(const Con<real>& c, const ModelT<MR>& m, const real* r, real* ua, real* ub) {
  const real* n = c.frame;
  real al[3], aa[3], t[3];
  for (int k = 0; k < 3; k++) { al[k] = m.mu * (n[k] - c.t.h.bw[k]); aa[k] = -m.mu * c.t.h.bw[3 + k]; }
  cross3(t, r, al);
  for (int k = 0; k < 3; k++) { ua[k] = al[k]; ua[3 + k] = t[k] + aa[k]; }
  cross3(t, r, c.t.h.bw);
  for (int k = 0; k < 3; k++) { ub[k] = c.t.h.bw[k]; ub[3 + k] = t[k] + c.t.h.bw[3 + k]; }
}
// diagonal block of one side (r = contact point relative to the bar's centre): H (packed lower 6x6) += T^T K T
template <typename real, typename MR> TB_FN void side_hessian(const Con<real>& c, const ModelT<MR>& m, const real* r, real* H) {
  const ConW<real> w = con_weights(c, m);
  const real* n = c.frame;
  const real dl = w.wl0 - w.wl1, da = w.wa3 - w.wa4;
  real cv[3];
  cross3(cv, r, n);
  const real rr = dot3(r, r);
  // lin-lin: w1 I + dl n n^T
  H[0] += w.wl1 + dl * n[0] * n[0]; H[1] += dl * n[1] * n[0]; H[2] += w.wl1 + dl * n[1] * n[1];
  H[3] += dl * n[2] * n[0]; H[4] += dl * n[2] * n[1]; H[5] += w.wl1 + dl * n[2] * n[2];
  // ang-lin (rows 3..5, cols 0..2): w1 [r]x + dl c n^T
  H[6] += dl * cv[0] * n[0];              H[7] += -w.wl1 * r[2] + dl * cv[0] * n[1]; H[8] += w.wl1 * r[1] + dl * cv[0] * n[2];
  H[10] += w.wl1 * r[2] + dl * cv[1] * n[0]; H[11] += dl * cv[1] * n[1];              H[12] += -w.wl1 * r[0] + dl * cv[1] * n[2];
  H[15] += -w.wl1 * r[1] + dl * cv[2] * n[0]; H[16] += w.wl1 * r[0] + dl * cv[2] * n[1]; H[17] += dl * cv[2] * n[2];
  // ang-ang: w1 (|r|^2 I - r r^T) + dl c c^T + w4 I + da n n^T
  const real dg = w.wl1 * rr + w.wa4;
  H[9] += dg - w.wl1 * r[0] * r[0] + dl * cv[0] * cv[0] + da * n[0] * n[0];
  H[13] += -w.wl1 * r[1] * r[0] + dl * cv[1] * cv[0] + da * n[1] * n[0];
  H[14] += dg - w.wl1 * r[1] * r[1] + dl * cv[1] * cv[1] + da * n[1] * n[1];
  H[18] += -w.wl1 * r[2] * r[0] + dl * cv[2] * cv[0] + da * n[2] * n[0];
  H[19] += -w.wl1 * r[2] * r[1] + dl * cv[2] * cv[1] + da * n[2] * n[1];
  H[20] += dg - w.wl1 * r[2] * r[2] + dl * cv[2] * cv[2] + da * n[2] * n[2];
  if (c.zone == ZONE_MIDDLE) {
    real ua[6], ub[6];
    cone_side(c, m, r, ua, ub);
    rank1_sym(H, c.t.h.ca, ua);
    rank1_sym(H, -c.t.h.cb, ub);
  }
}
// block between the two bars of a bar-bar contact: X (6x6 row-major, rows = bar with offset rh, cols = bar with rl)
// += -T_h^T K T_l   (the two sides enter J with opposite signs)
template <typename real, typename MR> TB_FN void cross_hessian(const Con<real>& c, const ModelT<MR>& m, const real* rh, const real* rl, real* X) {
  const ConW<real> w = con_weights(c, m);
  const real* n = c.frame;
  const real dl = w.wl0 - w.wl1, da = w.wa3 - w.wa4;
  real ch[3], cl[3];
  cross3(ch, rh, n); cross3(cl, rl, n);
  const real hl = dot3(rh, rl);
  // [r]x as a matrix: rows (0, -z, y), (z, 0, -x), (-y, x, 0)
  const real Sh[9] = {0, -rh[2], rh[1], rh[2], 0, -rh[0], -rh[1], rh[0], 0};
  const real Sl[9] = {0, -rl[2], rl[1], rl[2], 0, -rl[0], -rl[1], rl[0], 0};
  for (int i = 0; i < 3; i++)
    for (int k = 0; k < 3; k++) {
      const real id = i == k ? real(1) : real(0);
      // lin-lin: A = w1 I + dl n n^T
      X[6 * i + k] -= w.wl1 * id + dl * n[i] * n[k];
      // lin(h)-ang(l): A X_l = -w1 [r_l]x + dl n c_l^T
      X[6 * i + 3 + k] -= -w.wl1 * Sl[3 * i + k] + dl * n[i] * cl[k];
      // ang(h)-lin(l): X_h^T A = w1 [r_h]x + dl c_h n^T
      X[6 * (3 + i) + k] -= w.wl1 * Sh[3 * i + k] + dl * ch[i] * n[k];
      // ang-ang: w1 ((r_h . r_l) I - r_l r_h^T) + dl c_h c_l^T + w4 I + da n n^T
      X[6 * (3 + i) + 3 + k] -= w.wl1 * (hl * id - rl[i] * rh[k]) + dl * ch[i] * cl[k] + w.wa4 * id + da * n[i] * n[k];
    }
  if (c.zone == ZONE_MIDDLE) {
    real uah[6], ubh[6], ual[6], ubl[6];
    cone_side(c, m, rh, uah, ubh); cone_side(c, m, rl, ual, ubl);
    rank1_gen(X, -c.t.h.ca, uah, ual);
    rank1_gen(X, c.t.h.cb, ubh, ubl);
  }
}

// ---- 6x6 block kernels of the Newton solve on blocks in shared memory (packed lower triangles: entry (i, k) at
// i (i + 1) / 2 + k; full blocks row-major).  Each loads its operands into registers, works unrolled, stores back.
// A = L D L^T in place: strict lower part = unit L, diagonal = d; dinv = 1 / d
template <typename real> TB_FN void blk_ldl(real* Ag, real* dinvg) {
  real A[21], dinv[6];
  TB_UNROLL
  for (int e = 0; e < 21; e++) A[e] = Ag[e];
  TB_UNROLL
  for (int j = 0; j < 6; j++) {
    real s = A[j * (j + 1) / 2 + j];
    TB_UNROLL
    for (int k = 0; k < j; k++) {
      real t = A[j * (j + 1) / 2 + k];
      TB_UNROLL
      for (int q = 0; q < k; q++) t -= A[j * (j + 1) / 2 + q] * A[q * (q + 1) / 2 + q] * A[k * (k + 1) / 2 + q];
      real l = t * dinv[k];
      A[j * (j + 1) / 2 + k] = l;
      s -= l * t;
    }
    s = tmax(s, Lim<real>::MINVAL);
    A[j * (j + 1) / 2 + j] = s;
    dinv[j] = trcp(s);
  }
  TB_UNROLL
  for (int e = 0; e < 21; e++) Ag[e] = A[e];
  TB_UNROLL
  for (int j = 0; j < 6; j++) dinvg[j] = dinv[j];
}
template <typename real> TB_FN void blk_fwd(const real* L, real* x) {   // x <- L^-1 x   (x in registers)
  TB_UNROLL
  for (int i = 1; i < 6; i++) {
    real t = x[i];
    TB_UNROLL
    for (int k = 0; k < i; k++) t -= L[i * (i + 1) / 2 + k] * x[k];
    x[i] = t;
  }
}
template <typename real> TB_FN void blk_bwd(const real* L, real* x) {   // x <- L^-T x
  TB_UNROLL
  for (int i = 4; i >= 0; i--) {
    real t = x[i];
    TB_UNROLL
    for (int k = i + 1; k < 6; k++) t -= L[k * (k + 1) / 2 + i] * x[k];
    x[i] = t;
  }
}
// Row-split forms of X <- X L^-T D^-1 and C -= A diag(d) B^T: the three lanes of an env share a block operation, two
// rows each (r0 = 2 * bar), so the warp's instruction stream carries two rows instead of six.
// rows r0, r0 + 1 of X <- X L^-T D^-1 ; L (packed, unit lower) and dinv in registers
template <typename real> TB_FN void blk_trsm_rows2(real* Xg, const real* L, const real* dinv, int r0) {
  TB_UNROLL
  for (int rr = 0; rr < 2; rr++) {
    real* X = Xg + 6 * (r0 + rr);
    real u[6];
    TB_UNROLL
    for (int k = 0; k < 6; k++) {
      real t = X[k];
      TB_UNROLL
      for (int q = 0; q < k; q++) t -= u[q] * L[k * (k + 1) / 2 + q];
      u[k] = t;
    }
    TB_UNROLL
    for (int k = 0; k < 6; k++) X[k] = u[k] * dinv[k];
  }
}
// rows r0, r0 + 1 of C -= A diag(d) B^T ; B (full 6x6) and d in registers.  sym: C packed lower (entries j <= i only)
template <typename real> TB_FN void blk_mulsub_rows2(real* Cg, const real* Ag, const real* d, const real* Bm, bool sym, int r0) {
  TB_UNROLL
  for (int rr = 0; rr < 2; rr++) {
    const int i = r0 + rr;
    real ad[6];
    TB_UNROLL
    for (int k = 0; k < 6; k++) ad[k] = Ag[6 * i + k] * d[k];
    real* Crow = sym ? Cg + i * (i + 1) / 2 : Cg + 6 * i;
    TB_UNROLL
    for (int j = 0; j < 6; j++) {
      real sacc = 0;
      TB_UNROLL
      for (int k = 0; k < 6; k++) sacc += ad[k] * Bm[6 * j + k];
      if (!sym || j <= i) Crow[j] -= sacc;
    }
  }
}
template <typename real> TB_FN void blk_gemv_sub(real* y, const real* A, const real* x) {   // y -= A x   (y in registers)
  TB_UNROLL
  for (int i = 0; i < 6; i++) {
    real t = y[i];
    TB_UNROLL
    for (int k = 0; k < 6; k++) t -= A[6 * i + k] * x[k];
    y[i] = t;
  }
}
template <typename real> TB_FN void blk_gemvT_sub(real* y, const real* A, const real* x) {   // y -= A^T x
  TB_UNROLL
  for (int i = 0; i < 6; i++) {
    real t = y[i];
    TB_UNROLL
    for (int k = 0; k < 6; k++) t -= A[6 * k + i] * x[k];
    y[i] = t;
  }
}

// ------------------------------------------------------------------ collision pieces
template <typename real>
TB_NOINL void plane_cylinder_points(const ModelT<real>& m, const real* pos2, const real* axis_in, real radius, real half,
                                    const real* xaxis, int& cnt, real dist[4], real pts[4][3]) {
  const real* normal = m.fnormal;
  real axis[3], vec[3];
  copy3(axis, axis_in);
  real prjaxis = dot3(normal, axis);
  if (prjaxis > 0) { scl3(axis, axis, real(-1)); prjaxis = -prjaxis; }
  sub3(vec, pos2, m.fpos);
  real dist0 = dot3(vec, normal);
  scl3(vec, axis, prjaxis); sub3(vec, vec, normal);
  real len_sqr = dot3(vec, vec);
  if (len_sqr >= Lim<real>::MINVAL * Lim<real>::MINVAL) scl3(vec, vec, radius / tsqrt(len_sqr));
  else scl3(vec, xaxis, radius);
  real prjvec = dot3(vec, normal);
  scl3(axis, axis, half); prjaxis *= half;
  cnt = 0;
  if (dist0 + prjaxis + prjvec <= 0) {
    dist[cnt] = dist0 + prjaxis + prjvec;
    add3(pts[cnt], pos2, vec); add3(pts[cnt], pts[cnt], axis); addscl3(pts[cnt], normal, -dist[cnt] * real(0.5));
    cnt++;
  } else return;
  if (dist0 - prjaxis + prjvec <= 0) {
    dist[cnt] = dist0 - prjaxis + prjvec;
    add3(pts[cnt], pos2, vec); sub3(pts[cnt], pts[cnt], axis); addscl3(pts[cnt], normal, -dist[cnt] * real(0.5));
    cnt++;
  }
  real prjvec1 = -prjvec * real(0.5);
  if (dist0 + prjaxis + prjvec1 <= 0) {
    real vec1[3];
    cross3(vec1, vec, axis); normalize3(vec1); scl3(vec1, vec1, radius * tsqrt(real(3)) * real(0.5));
    for (int s = 0; s < 2; s++) {
      dist[cnt] = dist0 + prjaxis + prjvec1;
      add3(pts[cnt], pos2, axis); addscl3(pts[cnt], vec1, s ? real(-1) : real(1)); addscl3(pts[cnt], vec, real(-0.5));
      addscl3(pts[cnt], normal, -dist[cnt] * real(0.5));
      cnt++;
    }
  }
}
// squared distance between segments p1 +- a1, p2 +- a2 (a = half-axis vectors)
template <typename real> TB_FN real segseg_dist2(const real* p1, const real* a1, const real* p2, const real* a2) {
  real r[3]; sub3(r, p1, p2);
  real A = dot3(a1, a1), E = dot3(a2, a2), Bq = dot3(a1, a2), C = dot3(a1, r), F = dot3(a2, r);
  real den = A * E - Bq * Bq, s = 0, t;
  if (den > real(1e-30)) s = clampr(tdiv(Bq * F - C * E, den), real(-1), real(1));
  t = tdiv(Bq * s + F, E);
  if (t < real(-1)) { t = real(-1); s = clampr(tdiv(-Bq - C, A), real(-1), real(1)); }
  else if (t > real(1)) { t = real(1); s = clampr(tdiv(Bq - C, A), real(-1), real(1)); }
  real d[3] = {r[0] + s * a1[0] - t * a2[0], r[1] + s * a1[1] - t * a2[1], r[2] + s * a1[2] - t * a2[2]};
  return dot3(d, d);
}
template <typename real> TB_FN real ptseg_dist2(const real* c, const real* p, const real* a) {
  real r[3]; sub3(r, c, p);
  real t = clampr(tdiv(dot3(r, a), dot3(a, a)), real(-1), real(1));
  addscl3(r, a, -t);
  return dot3(r, r);
}

// height-field prism k of row r (vertices n = k, k+1, k+2 of the strip; c = cmin + n/2, odd n -> row r, even -> r + 1)
template <typename real> TB_FN void hf_prism(const ModelT<real>& m, int r, int cmin, int k, CObj<real>& o) {
  for (int j = 0; j < 3; j++) {
    int n = k + j, c = cmin + n / 2, rr = r + ((n & 1) ? 0 : 1);
    o.px[j] = m.hdx * c - m.hsize[0]; o.py[j] = m.hdy * rr - m.hsize[1];
    o.pz[j] = (real)m.hdata[rr * m.ncol + c] * m.hsize[2];
  }
  o.pbase = -m.hsize[3];
}
// Conservative cull before MPR: a prism lies on or below the plane through its three top vertices, so a geom whose
// support point towards that plane stays above it (by more than a rounding slack) cannot touch the prism.
template <typename real>
TB_FN bool hf_above_top_plane(const CObj<real>& pr, int gtype, const real* pos, const real* R, real rad, real hl) {
  real e1[3] = {pr.px[1] - pr.px[0], pr.py[1] - pr.py[0], pr.pz[1] - pr.pz[0]};
  real e2[3] = {pr.px[2] - pr.px[0], pr.py[2] - pr.py[0], pr.pz[2] - pr.pz[0]};
  real n[3];
  cross3(n, e1, e2);
  if (n[2] < 0) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }
  real nn = dot3(n, n);
  if (!(nn > 0)) return false;
  real reach;
  if (gtype == GEOM_SPHERE) reach = rad * tsqrt(nn);
  else {
    real na = n[0] * R[2] + n[1] * R[5] + n[2] * R[8];
    reach = hl * tabs(na) + rad * tsqrt(tmax(real(0), nn - na * na));
  }
  real top0[3] = {pr.px[0], pr.py[0], pr.pz[0]};
  real sep = dot3(n, pos) - reach - dot3(n, top0);
  return sep > real(1e-9) * tsqrt(nn);
}

// stores a new active contact of this lane (dist >= 0 gives no rows: includemargin 0)
template <typename P>
TB_FN void add_contact(EnvSh<P>& S, int lane_bar, int& nmine, int b1, int b2, typename P::real dist, const typename P::real* pos,
                       const typename P::real* normal) {
  typedef typename P::sreal sreal;
  if (!(dist < 0)) return;
  if (nmine >= MAXCL) { S.overflow = 1; return; }
  Con<sreal>& c = con_of(S, lane_bar, nmine++);
  c.b1 = b1; c.b2 = b2; c.owner = lane_bar;
  for (int k = 0; k < 3; k++) c.frame[k] = (sreal)normal[k];
  make_frame(c.frame);
  for (int k = 0; k < 3; k++) {
    c.r2[k] = (sreal)pos[k] - (sreal)S.xpos[3 * b2 + k];
    c.r1[k] = b1 >= 0 ? (sreal)pos[k] - (sreal)S.xpos[3 * b1 + k] : sreal(0);
  }
  c.D0 = (sreal)dist;   // parked until the rows are built
}

// ------------------------------------------------------------------ the stages of one physics pass
// Every stage is entered by all 32 lanes of the warp with per-lane predicates (`on`, `act`, `go`: does this lane's env
// take part), the same convention as tb_env.cuh.  Stages may exchange data within the warp (wsync, any, sum3, grp_any)
// but contain no CTA barrier: every uni_any is in phys(), so that the rule "every warp of a CTA makes the same sequence
// of these calls" can be checked in one function.  Per-lane arrays that cross stages are grouped in the two structs
// below and indexed only with indices that are constant after unrolling (a dynamically indexed per-thread array would
// live in local memory).

// the bar's rotation matrix, in the collision precision and in the solver precision
template <typename P> struct BarFrame { typename P::real R[9]; typename P::sreal Rs[9]; };
// the bar's 6-vectors of the constraint solve, angular parts in WORLD-frame components: asm_ = qacc_smooth, Iw = the
// rotational inertia R diag(I) R^T (packed lower), fcon = the constraint wrench
template <typename P> struct BarSolve { typename P::sreal asm_[6], Iw[6], fcon[6]; };

// publishes a per-bar 6-vector (a world-frame twist) for the contact owners
template <typename P> TB_FN void publish(EnvSh<P>& S, int b, const typename P::sreal* a, bool doit) {
  if (doit) for (int k = 0; k < 6; k++) S.u.sol.xv[6 * b + k] = a[k];
}
// out = M_w d for this bar (mass on the linear part, world-frame rotational inertia on the angular part)
template <typename P>
TB_FN void mulM(const ModelT<typename P::real>& m, int b, const BarSolve<P>& N, const typename P::sreal* d, typename P::sreal* out) {
  typedef typename P::sreal sreal;
  const typename P::real* Mb = m.M + 6 * b;
  for (int k = 0; k < 3; k++) out[k] = (sreal)Mb[k] * d[k];
  out[3] = N.Iw[0] * d[3] + N.Iw[1] * d[4] + N.Iw[3] * d[5];
  out[4] = N.Iw[1] * d[3] + N.Iw[2] * d[4] + N.Iw[4] * d[5];
  out[5] = N.Iw[3] * d[3] + N.Iw[4] * d[4] + N.Iw[5] * d[5];
}

// mj_resetData on this lane's bar
template <typename P> TB_FN void reset_bar(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, int b) {
  for (int k = 0; k < 3; k++) B.x[k] = m.qpos0[7 * b + k];
  for (int k = 0; k < 4; k++) B.q[k] = m.qpos0[7 * b + 3 + k];
  for (int k = 0; k < 6; k++) { B.v[k] = 0; B.warm[k] = 0; }
  if (b == 0) for (int k = 0; k < NACT; k++) { S.ctrl[k] = 0; S.act[k] = 0; }
}

// mj_checkPos / mj_checkVel: an env with a non-finite position or velocity is reset
template <typename P> TB_FN void check_state(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, const LaneCtx& L, bool on) {
  bool bad = false;
  for (int k = 0; k < 3; k++) bad |= is_bad(B.x[k]);
  for (int k = 0; k < 4; k++) bad |= is_bad(B.q[k]);
  for (int k = 0; k < 6; k++) bad |= is_bad(B.v[k]);
  bad = grp_any(bad && on, L.base);
  if (bad && on) { if (L.bar == 0) S.bad |= 1; reset_bar(B, S, m, L.bar); }
  wsync();
}

// kinematics: the bar's frame, and its pose, world twist, end-cap centres and tendon sites in shared memory
template <typename P>
TB_FN void kinematics(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, int b, BarFrame<P>& F, bool on) {
  typedef typename P::real real; typedef typename P::sreal sreal;
  if (!on) return;
  normalize4(B.q);
  quat2mat(F.R, B.q);
  for (int k = 0; k < 9; k++) F.Rs[k] = (sreal)F.R[k];
  for (int k = 0; k < 3; k++) { S.xpos[3 * b + k] = B.x[k]; S.vw[6 * b + k] = B.v[k]; }
  for (int k = 0; k < 9; k++) S.xmat[9 * b + k] = F.R[k];
  real ww[3];
  mulMV(ww, F.R, B.v + 3);
  for (int k = 0; k < 3; k++) S.vw[6 * b + 3 + k] = ww[k];
  for (int i = 0; i < 2; i++) {   // end-cap centres s(2b), s(2b+1): geoms 1, 2 of the bar
    real c[3];
    mulMV(c, F.R, m.gpos[5 * b + 1 + i]);
    for (int k = 0; k < 3; k++) S.sph[3 * (2 * b + i) + k] = B.x[k] + c[k];
  }
  for (int n = 0; n < m.nends[b]; n++) {
    int end = m.ends[b][n];
    real c[3];
    mulMV(c, F.R, m.tsite[end]);
    for (int k = 0; k < 3; k++) S.u.site[3 * end + k] = B.x[k] + c[k];
  }
}

// Tendon and actuator constants of the per-env variant, read from the env's row with the (real) cast make_model uses,
// so that the nominal row reproduces the model bit for bit.  Plain loads, not __ldg: a reset writes the row in the
// same launch (run_reset, run_pool).  The accessors hand the default variant the model's fields, read where the code
// always read them.
template <typename P> struct PrmRow { typename P::real tk, tdamp, tls[2], gain, bias[3], dynprm0; };
template <typename P> TB_FN void load_act_prm(PrmRow<P>& R, const double* r) {
  typedef typename P::real real;
  R.gain = (real)r[PRM_GAIN];
  for (int k = 0; k < 3; k++) R.bias[k] = (real)r[PRM_BIAS + k];
  R.dynprm0 = (real)r[PRM_DYNPRM0];
}
template <typename P> TB_FN void load_ten_prm(PrmRow<P>& R, const double* r, int t) {
  typedef typename P::real real;
  R.tk = (real)r[PRM_TK + t]; R.tdamp = (real)r[PRM_TDAMP + t];
  R.tls[0] = (real)r[PRM_TLS + 2 * t]; R.tls[1] = (real)r[PRM_TLS + 2 * t + 1];
}
template <typename P> TB_FN typename P::real prm_tk(const PrmRow<P>& R, const ModelT<typename P::real>& m, int t) {
  if constexpr (P::per_env) return R.tk; else return m.tk[t];
}
template <typename P> TB_FN typename P::real prm_tdamp(const PrmRow<P>& R, const ModelT<typename P::real>& m, int t) {
  if constexpr (P::per_env) return R.tdamp; else return m.tdamp[t];
}
template <typename P> TB_FN typename P::real prm_tls(const PrmRow<P>& R, const ModelT<typename P::real>& m, int t, int k) {
  if constexpr (P::per_env) return R.tls[k]; else return m.tls[t][k];
}
template <typename P> TB_FN typename P::real prm_gain(const PrmRow<P>& R, const ModelT<typename P::real>& m) {
  if constexpr (P::per_env) return R.gain; else return m.gain;
}
template <typename P> TB_FN typename P::real prm_bias(const PrmRow<P>& R, const ModelT<typename P::real>& m, int k) {
  if constexpr (P::per_env) return R.bias[k]; else return m.bias[k];
}
template <typename P> TB_FN typename P::real prm_dynprm0(const PrmRow<P>& R, const ModelT<typename P::real>& m) {
  if constexpr (P::per_env) return R.dynprm0; else return m.dynprm0;
}

// tendons: length, velocity, spring-damper / actuator force; then qacc_smooth, the world-frame inertia, and the damping
// block Dblk of the bar (for implicitfast)
template <typename P>
TB_FN void smooth_dynamics(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, int b, const BarFrame<P>& F,
                           BarSolve<P>& N, typename P::real* Dblk, bool on) {
  typedef typename P::real real; typedef typename P::sreal sreal;
  if (!on) return;
  const real MINV = Lim<real>::MINVAL;
  const real* Mb = m.M + 6 * b;
  real f[6] = {0, 0, 0, 0, 0, 0};
  for (int e = 0; e < 21; e++) Dblk[e] = 0;
  PrmRow<P> R;
  if constexpr (P::per_env) load_act_prm(R, S.prm);
  TB_UNROLL1
  for (int n = 0; n < m.nends[b]; n++) {
    const int end = m.ends[b][n], t = end >> 1, s = end & 1, oe = end ^ 1, ob = m.tbody[oe];
    if constexpr (P::per_env) load_ten_prm(R, S.prm, t);
    real pown[3], poth[3], dir[3];
    copy3(pown, S.u.site + 3 * end); copy3(poth, S.u.site + 3 * oe);
    if (s) sub3(dir, pown, poth); else sub3(dir, poth, pown);
    real len = normalize3(dir);
    real ro[3], co[3], cw[3], Jw[3];
    sub3(ro, pown, B.x); cross3(co, ro, dir); mulMTV(Jw, F.R, co);
    real vown = dot3(dir, B.v) + dot3(Jw, B.v + 3);
    sub3(ro, poth, S.xpos + 3 * ob); cross3(cw, ro, dir);
    real voth = dot3(dir, S.vw + 6 * ob) + dot3(cw, S.vw + 6 * ob + 3);
    real vel = s ? (vown - voth) : (voth - vown);
    real frc = 0, Bt = -prm_tdamp(R, m, t);
    if (prm_tk(R, m, t) > 0) {
      if (len > prm_tls(R, m, t, 1)) frc = prm_tk(R, m, t) * (prm_tls(R, m, t, 1) - len);
      else if (len < prm_tls(R, m, t, 0)) frc = prm_tk(R, m, t) * (prm_tls(R, m, t, 0) - len);
    }
    frc -= prm_tdamp(R, m, t) * vel;
    const int a = m.ten_act[t];
    if (a >= 0) {
      real ctrl = (real)S.ctrl[a], input;
      if (m.ctrllimited) ctrl = clampr(ctrl, m.ctrlrange[0], m.ctrlrange[1]);
      real act = (real)S.act[a];
      if (m.dyntype) { if (s == 0) S.actdot[a] = (ctrl - act) / tmax(MINV, prm_dynprm0(R, m)); input = act; }
      else { if (s == 0) S.actdot[a] = 0; input = ctrl; }
      real fa = prm_gain(R, m) * input + prm_bias(R, m, 0) + prm_bias(R, m, 1) * len + prm_bias(R, m, 2) * vel;
      bool clamped = false;
      if (m.forcelimited) {
        clamped = (fa <= m.forcerange[0] || fa >= m.forcerange[1]);
        fa = clampr(fa, m.forcerange[0], m.forcerange[1]);
      }
      frc += fa;
      if (prm_bias(R, m, 2) != 0 && ((m.flags & 1u) || !clamped)) Bt += prm_bias(R, m, 2);
    }
    if (s == 0) S.tlen[t] = len;
    real sg = s ? frc : -frc;
    real j[6] = {dir[0], dir[1], dir[2], Jw[0], Jw[1], Jw[2]};
    for (int k = 0; k < 6; k++) f[k] += sg * j[k];
    rank1_sym(Dblk, Bt, j);
  }
  // qacc_smooth = M^-1 (passive + actuator - bias)
  const real* I = m.inertia[b];
  const real* w = B.v + 3;
  sreal al[3];
  for (int k = 0; k < 3; k++) {
    int k1 = (k + 1) % 3, k2 = (k + 2) % 3;
    N.asm_[k] = (sreal)((f[k] + Mb[k] * m.grav[k]) * m.invM[6 * b + k]);
    al[k] = (sreal)((f[3 + k] - (w[k1] * (I[k2] * w[k2]) - w[k2] * (I[k1] * w[k1]))) * m.invM[6 * b + 3 + k]);
  }
  // from here to the end of the solve the bar's angular dofs are WORLD-frame components (the rotation is orthogonal,
  // so costs, norms and the Newton direction are the same as in body coordinates): qacc_smooth, the warm start /
  // iterate, and the rotational inertia R diag(I) R^T
  mulMV(N.asm_ + 3, F.Rs, al);
  mulMV(al, F.Rs, B.warm + 3);
  for (int k = 0; k < 3; k++) B.warm[3 + k] = al[k];
  for (int i = 0, e = 0; i < 3; i++)
    for (int k = 0; k <= i; k++, e++)
      N.Iw[e] = F.Rs[3 * i] * (sreal)I[0] * F.Rs[3 * k] + F.Rs[3 * i + 1] * (sreal)I[1] * F.Rs[3 * k + 1] + F.Rs[3 * i + 2] * (sreal)I[2] * F.Rs[3 * k + 2];
}

// plane collision of the bar's five geoms
template <typename P>
TB_FN void collide_plane(const BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, int b, const BarFrame<P>& F, int& nmine, bool on) {
  typedef typename P::real real;
  if (!on) return;
  const real* R = F.R;
  TB_UNROLL1
  for (int g = 0; g < 5; g++) {
    const int Gi = 5 * b + g;
    real c[3], tmp[3];
    for (int k = 0; k < 3; k++) c[k] = B.x[k] + R[3 * k + 2] * m.gz[Gi];
    sub3(tmp, c, m.fpos);
    real cdist = dot3(tmp, m.fnormal);
    if (m.gtype[Gi] == GEOM_SPHERE) {
      real r = m.gsize[Gi][0];
      if (cdist <= r) {
        real dist = cdist - r, pos[3];
        copy3(pos, c); addscl3(pos, m.fnormal, -dist / 2 - r);
        add_contact(S, b, nmine, -1, b, dist, pos, m.fnormal);
      }
    } else if (cdist <= m.gbound[Gi]) {
      real axis[3] = {R[2], R[5], R[8]}, xaxis[3] = {R[0], R[3], R[6]}, dist[4], pts[4][3];
      int cnt = 0;
      plane_cylinder_points(m, c, axis, m.gsize[Gi][0], m.gsize[Gi][1], xaxis, cnt, dist, pts);
      for (int k = 0; k < cnt; k++) add_contact(S, b, nmine, -1, b, dist[k], pts[k], m.fnormal);
    }
  }
}

// height field (frame axis-aligned at fpos).  Pass 1: per geom, the prisms under its AABB whose top reaches the AABB's
// bottom (MuJoCo's test) and that the geom can reach (conservative cull) are listed in a bit mask, kept with the geom's
// cell window in the env's solver scratch (idle until the Newton stage, behind the lanes' MPR objects).  Pass 2: the
// lanes of the warp take their candidates through MPR round by round, together, each lane walking its own geoms in
// order -- the number of rounds is the largest candidate count of a LANE, not the sum over the five geoms of the
// largest count per geom, and the contacts are found in the same order.
template <typename P>
TB_FN void collide_hfield(const BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, int b, const BarFrame<P>& F,
                          int& nmine, int& nmpr, bool on) {
  typedef typename P::real real; typedef typename P::sreal sreal;
  const real MINV = Lim<real>::MINVAL;
  const real* R = F.R;
  int* hfc = reinterpret_cast<int*>(&S.u.sol.D[0][0]) + 240 + 20 * b;   // [geom][mask, cmin, rmin, per_row]
  static_assert(6 * sizeof(CObj<sreal>) <= 960 && (240 + 60) * sizeof(int) <= sizeof(S.u.sol.D) + sizeof(S.u.sol.O), "solver scratch too small");
  TB_UNROLL1
  for (int g = 0; g < 5; g++) {
    const int Gi = 5 * b + g;
    unsigned cand = 0;
    int cmin = 0, rmin = 0, per_row = 1;
    real pos[3];
    for (int k = 0; k < 3; k++) pos[k] = B.x[k] + R[3 * k + 2] * m.gz[Gi] - m.fpos[k];
    const real r = m.gsize[Gi][0], hl = m.gsize[Gi][1], rb = m.gbound[Gi];
    if (on) {
      bool ok = true;
      for (int i = 0; i < 2; i++) if (m.hsize[i] < pos[i] - rb || -m.hsize[i] > pos[i] + rb) ok = false;
      if (m.hsize[2] < pos[2] - rb || -m.hsize[3] > pos[2] + rb) ok = false;
      real ext[3];
      if (m.gtype[Gi] == GEOM_SPHERE) ext[0] = ext[1] = ext[2] = r;
      else for (int i = 0; i < 3; i++) {   // AABB half extents of a cylinder = what the +-axis support queries return
        real az = R[3 * i + 2];
        ext[i] = r * tsqrt(tmax(real(0), 1 - az * az)) + hl * tabs(az);
      }
      real xmin = pos[0] - ext[0], xmax = pos[0] + ext[0], ymin = pos[1] - ext[1], ymax = pos[1] + ext[1];
      real zmin = pos[2] - ext[2], zmax = pos[2] + ext[2];
      if (xmin > m.hsize[0] || xmax < -m.hsize[0] || ymin > m.hsize[1] || ymax < -m.hsize[1] || zmin > m.hsize[2] || zmax < -m.hsize[3]) ok = false;
      if (ok) {
        cmin = (int)tfloor((xmin + m.hsize[0]) / (2 * m.hsize[0]) * (m.ncol - 1));
        int cmax = (int)tceil((xmax + m.hsize[0]) / (2 * m.hsize[0]) * (m.ncol - 1));
        rmin = (int)tfloor((ymin + m.hsize[1]) / (2 * m.hsize[1]) * (m.nrow - 1));
        int rmax = (int)tceil((ymax + m.hsize[1]) / (2 * m.hsize[1]) * (m.nrow - 1));
        if (cmin < 0) cmin = 0;
        if (cmax > m.ncol - 1) cmax = m.ncol - 1;
        if (rmin < 0) rmin = 0;
        if (rmax > m.nrow - 1) rmax = m.nrow - 1;
        per_row = 2 * (cmax - cmin + 1) - 2;
        if (per_row > 0 && rmax > rmin) {
          if (per_row * (rmax - rmin) > 32) S.overflow = 1;
          TB_UNROLL1
          for (int q = 0; q < per_row * (rmax - rmin) && q < 32; q++) {
            CObj<real> o1;
            hf_prism(m, rmin + q / per_row, cmin, q % per_row, o1);
            if (!(o1.pz[0] >= zmin || o1.pz[1] >= zmin || o1.pz[2] >= zmin)) continue;
            if (hf_above_top_plane(o1, m.gtype[Gi], pos, R, r, hl)) continue;
            cand |= 1u << q;
          }
        } else per_row = 1;
      }
      hfc[4 * g] = (int)cand; hfc[4 * g + 1] = cmin; hfc[4 * g + 2] = rmin; hfc[4 * g + 3] = per_row;
    }
  }
  int g = -1, cmin = 0, rmin = 0, per_row = 1;
  unsigned cand = 0;
  TB_UNROLL1
  for (;;) {
    if (on) while (cand == 0 && g < 4) { g++; cand = (unsigned)hfc[4 * g]; cmin = hfc[4 * g + 1]; rmin = hfc[4 * g + 2]; per_row = hfc[4 * g + 3]; }
    const bool has = on && cand != 0;
    if (!any(has)) break;
    // the narrow phase runs in the solver's precision: MPR's 1e-6 tolerance is out of fp32's reach.  The lane's two
    // objects live in the env's solver scratch, not in per-thread local memory; only lanes with a candidate write
    // them (the idle lanes 30, 31 alias the last env's slice)
    CObj<sreal>* objs = reinterpret_cast<CObj<sreal>*>(&S.u.sol.D[0][0]) + 2 * b;
    CObj<sreal>&o1 = objs[0], &o2 = objs[1];
    real gc[3] = {0, 0, 0};
    if (has) {
      const int Gi = 5 * b + g;
      const int q = lowbit(cand);
      cand &= cand - 1;
      CObj<real> pr;
      hf_prism(m, rmin + q / per_row, cmin, q % per_row, pr);
      o1.type = 100;
      for (int k = 0; k < 3; k++) { o1.px[k] = pr.px[k]; o1.py[k] = pr.py[k]; o1.pz[k] = pr.pz[k]; }
      o1.pbase = pr.pbase;
      o2.type = m.gtype[Gi]; o2.size[0] = m.gsize[Gi][0]; o2.size[1] = m.gsize[Gi][1];
      for (int k = 0; k < 3; k++) { gc[k] = B.x[k] + R[3 * k + 2] * m.gz[Gi]; o2.pos[k] = gc[k] - m.fpos[k]; }
      for (int k = 0; k < 3; k++) o2.axis[k] = R[3 * k + 2];
      nmpr++;
    }
    sreal depthS = 0, dirS[3] = {0, 0, 1}, cpS[3] = {0, 0, 0};
    bool hit = mpr_penetration(o1, o2, (sreal)m.mpr_tol, m.mpr_iterations, has, &depthS, dirS, cpS);
    real depth = (real)depthS, dir[3] = {(real)dirS[0], (real)dirS[1], (real)dirS[2]}, cp[3] = {(real)cpS[0], (real)cpS[1], (real)cpS[2]};
    if (has) {
      if (hit && ccd_vec_is_origin(dir)) hit = false;
      if (hit) {
        add3(cp, cp, m.fpos);
        if ((m.flags & 4u) && o2.type == GEOM_SPHERE) {
          real nn[3]; sub3(nn, gc, cp);
          if (tsqrt(dot3(nn, nn)) > MINV) { normalize3(nn); copy3(dir, nn); }
        }
        add_contact(S, b, nmine, -1, b, -depth, cp, dir);
      }
    }
  }
}

// bar-bar: this lane takes pair p = its bar index: (0,1), (0,2), (1,2).  All geoms lie on their bar's axis, so the 25
// geom pairs are filtered with scalars: MuJoCo's bounding-sphere test, then an analytic capsule bound (conservative:
// MPR reports penetration only for intersecting shapes).  Sphere-sphere pairs are analytic; the others are listed in
// a bit mask and the lanes of the warp take their candidates through MPR round by round, together.
template <typename P>
TB_FN void collide_bars(EnvSh<P>& S, const ModelT<typename P::real>& m, int b, int& nmine, int& nmpr, bool on) {
  typedef typename P::real real; typedef typename P::sreal sreal;
  const real MINV = Lim<real>::MINVAL;
  const int pb1 = b == 2 ? 1 : 0, pb2 = b == 0 ? 1 : 2;
  const real *X1 = S.xpos + 3 * pb1, *X2 = S.xpos + 3 * pb2, *R1 = S.xmat + 9 * pb1, *R2 = S.xmat + 9 * pb2;
  unsigned cand = 0;
  if (on) {
    const real a1[3] = {R1[2], R1[5], R1[8]}, a2[3] = {R2[2], R2[5], R2[8]};
    real D[3]; sub3(D, X1, X2);
    const real DD = dot3(D, D), Da1 = dot3(D, a1), Da2 = dot3(D, a2), a12 = dot3(a1, a2);
    TB_UNROLL1
    for (int i = 0; i < 25; i++) {
      const int g1 = 5 * pb1 + i / 5, g2 = 5 * pb2 + i % 5;
      const real z1 = m.gz[g1], z2 = m.gz[g2];
      // centre difference r = D + z1 a1 - z2 a2
      const real rr = DD + z1 * z1 + z2 * z2 + 2 * (z1 * Da1 - z2 * Da2 - z1 * z2 * a12);
      const real bs = m.gbound[g1] + m.gbound[g2];
      if (rr > bs * bs) continue;   // MuJoCo's own bounding-sphere test
      const int t1 = m.gtype[g1], t2 = m.gtype[g2];
      const real rs = m.gsize[g1][0] + m.gsize[g2][0] + real(1e-6), h1 = m.gsize[g1][1], h2 = m.gsize[g2][1];
      const real ra1 = Da1 + z1 - z2 * a12, ra2 = Da2 + z1 * a12 - z2;   // a1 . r, a2 . r
      real d2;
      if (t1 == GEOM_SPHERE && t2 == GEOM_SPHERE) d2 = rr;
      else if (t1 == GEOM_SPHERE) { real t = clampr(tdiv(ra2, h2), real(-1), real(1)); d2 = rr - 2 * t * h2 * ra2 + t * t * h2 * h2; }
      else if (t2 == GEOM_SPHERE) { real t = clampr(tdiv(-ra1, h1), real(-1), real(1)); d2 = rr + 2 * t * h1 * ra1 + t * t * h1 * h1; }
      else {
        const real A = h1 * h1, E = h2 * h2, Bq = h1 * h2 * a12, C = h1 * ra1, F = h2 * ra2;
        real den = A * E - Bq * Bq, sg = 0, t;
        if (den > real(1e-30)) sg = clampr(tdiv(Bq * F - C * E, den), real(-1), real(1));
        t = tdiv(Bq * sg + F, E);
        if (t < real(-1)) { t = real(-1); sg = clampr(tdiv(-Bq - C, A), real(-1), real(1)); }
        else if (t > real(1)) { t = real(1); sg = clampr(tdiv(Bq - C, A), real(-1), real(1)); }
        d2 = rr + sg * sg * A + t * t * E + 2 * (sg * C - t * F - sg * t * Bq);
      }
      if (!(d2 <= rs * rs)) continue;
      if (t1 == GEOM_SPHERE && t2 == GEOM_SPHERE) {
        real c1[3], c2[3], nrm[3], pos[3];
        for (int k = 0; k < 3; k++) { c1[k] = X1[k] + a1[k] * z1; c2[k] = X2[k] + a2[k] * z2; }
        sub3(nrm, c2, c1);
        real len = normalize3(nrm), r1 = m.gsize[g1][0], dist = len - r1 - m.gsize[g2][0];
        nmpr++;
        copy3(pos, c1); addscl3(pos, nrm, r1 + dist / 2);
        if (dist <= 0) add_contact(S, b, nmine, pb1, pb2, dist, pos, nrm);
      } else cand |= 1u << i;
    }
  }
  TB_UNROLL1
  while (any(cand != 0)) {
    const bool has = cand != 0;
    int cb1 = pb1, cb2 = pb2;
    CObj<sreal>* objs = reinterpret_cast<CObj<sreal>*>(&S.u.sol.D[0][0]) + 2 * b;
    CObj<sreal>&o1 = objs[0], &o2 = objs[1];
    if (has) {
      const int i = lowbit(cand);
      cand &= cand - 1;
      int g1 = 5 * pb1 + i / 5, g2 = 5 * pb2 + i % 5;
      const real *Ra = R1, *Rb = R2, *Xa = X1, *Xb = X2;
      if (m.gtype[g1] > m.gtype[g2]) {   // lower geom type first
        int ti = g1; g1 = g2; g2 = ti; cb1 = pb2; cb2 = pb1;
        Ra = R2; Rb = R1; Xa = X2; Xb = X1;
      }
      o1.type = m.gtype[g1]; o1.size[0] = m.gsize[g1][0]; o1.size[1] = m.gsize[g1][1];
      o2.type = m.gtype[g2]; o2.size[0] = m.gsize[g2][0]; o2.size[1] = m.gsize[g2][1];
      for (int k = 0; k < 3; k++) { o1.axis[k] = Ra[3 * k + 2]; o2.axis[k] = Rb[3 * k + 2]; }
      for (int k = 0; k < 3; k++) { o1.pos[k] = Xa[k] + Ra[3 * k + 2] * m.gz[g1]; o2.pos[k] = Xb[k] + Rb[3 * k + 2] * m.gz[g2]; }
      nmpr++;
    }
    sreal depthS = 0, nrmS[3] = {1, 0, 0}, posS[3] = {0, 0, 0};
    bool hit = mpr_penetration(o1, o2, (sreal)m.mpr_tol, m.mpr_iterations, has, &depthS, nrmS, posS);
    real depth = (real)depthS, nrm[3] = {(real)nrmS[0], (real)nrmS[1], (real)nrmS[2]}, pos[3] = {(real)posS[0], (real)posS[1], (real)posS[2]};
    if (has) {
      if (hit && ccd_vec_is_origin(nrm)) hit = false;
      if (hit && (m.flags & 4u) && o1.type == GEOM_SPHERE) {
        real nn[3] = {pos[0] - (real)o1.pos[0], pos[1] - (real)o1.pos[1], pos[2] - (real)o1.pos[2]};
        if (tsqrt(dot3(nn, nn)) > MINV) { normalize3(nn); copy3(nrm, nn); }
      }
      if (hit) add_contact(S, b, nmine, cb1, cb2, -depth, pos, nrm);
    }
  }
}

// rows of this lane's contacts: velocity, impedance, reference acceleration, residual at qacc_smooth.  Returns the
// lane's part of the constraint cost at qacc_smooth; bbmine: does this lane own a bar-bar contact
template <typename P>
TB_FN typename P::sreal contact_rows(EnvSh<P>& S, const ModelT<typename P::real>& m, int b, int nmine, bool on, bool& bbmine) {
  typedef typename P::sreal sreal;
  const sreal SMINV = Lim<sreal>::MINVAL;
  sreal csm = 0;
  bbmine = false;
  if (on && nmine > 0) {
    TB_UNROLL1
    for (int s = 0; s < nmine; s++) {
      Con<sreal>& c = con_of(S, b, s);
      sreal dist = c.D0, vel[6], ja[6];
      con_mulJ(c, S.vw, vel);
      con_mulJ(c, S.u.sol.xv, ja);
      sreal imp = impedance(m, dist);
      sreal tran = (c.b1 >= 0 ? (sreal)m.invw_tran[c.b1] : sreal(0)) + (sreal)m.invw_tran[c.b2];
      c.D0 = trcp(tmax(SMINV, tdiv(1 - imp, imp) * tran));
      for (int r = 0; r < 6; r++) c.jar[r] = ja[r] - (-(sreal)m.B * vel[r] - (r ? sreal(0) : (sreal)m.K * imp * dist));
      csm += con_update(c, m, false, false);
      if (c.b1 >= 0) bbmine = true;
    }
  }
  return csm;
}

// mj_fwdConstraint's warm-start choice: the Newton iterate (B.warm) starts from the warm start or from qacc_smooth,
// whichever has the lower total cost (csm: this lane's part of the constraint cost at qacc_smooth)
template <typename P>
TB_FN void warm_start(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, const LaneCtx& L, const BarSolve<P>& N,
                      int nmine, typename P::sreal csm, bool act, bool on) {
  typedef typename P::sreal sreal;
  const int b = L.bar, base = L.base;
  bool use_smooth = false;
  if (any(act)) {
    wsync();
    sreal dw[6];
    for (int k = 0; k < 6; k++) dw[k] = B.warm[k] - N.asm_[k];
    publish(S, b, dw, act);
    wsync();
    sreal cws = 0;
    if (act) {
      if (nmine > 0) {
        TB_UNROLL1
        for (int s = 0; s < nmine; s++) {
          Con<sreal>& c = con_of(S, b, s);
          con_mulJ(c, S.u.sol.xv, c.jv);
          cws += con_update(c, m, false, true);
        }
      }
      sreal md[6];
      mulM(m, b, N, dw, md);
      for (int k = 0; k < 6; k++) cws += sreal(0.5) * md[k] * dw[k];
    }
    csm = sum3(csm, base); cws = sum3(cws, base);
    use_smooth = cws > csm;
    if (act && !use_smooth && nmine > 0) {
      TB_UNROLL1
      for (int s = 0; s < nmine; s++) {
        Con<sreal>& c = con_of(S, b, s);
        for (int r = 0; r < 6; r++) c.jar[r] += c.jv[r];
      }
    }
  }
  if (on) { if (!act || use_smooth) for (int k = 0; k < 6; k++) B.warm[k] = N.asm_[k]; }
}

// Newton: contact forces at the iterate (owners), then each bar lane gathers the wrenches of the contacts that touch
// its bar into N.fcon and forms the gradient.  Returns the env's total cost; gn: the squared norm of its gradient
template <typename P>
TB_FN typename P::sreal newton_gradient(const BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, const LaneCtx& L,
                                        BarSolve<P>& N, int nmine, int ngr, bool act, typename P::sreal* grad, typename P::sreal& gn) {
  typedef typename P::sreal sreal;
  const int b = L.bar, base = L.base;
  sreal cpart = 0;
  if (act && nmine > 0) {
    TB_UNROLL1
    for (int s = 0; s < nmine; s++) {
      Con<sreal>& c = con_of(S, b, s);
      cpart += con_update(c, m, true, false);
    }
  }
  wsync();
  gn = 0;
  if (act) {
    sreal Fw[3] = {0, 0, 0}, Tw[3] = {0, 0, 0};
    // own ground contacts (every lane on its own list: full lanes), then the bar-bar contacts of all three owners
    TB_UNROLL1
    for (int s = 0; s < ngr; s++) {
      const Con<sreal>& c = con_of(S, b, s);
      if (c.zone == ZONE_TOP) continue;
      sreal t[3];
      cross3(t, c.r2, c.wr);
      for (int k = 0; k < 3; k++) { Fw[k] += c.wr[k]; Tw[k] += t[k] + c.wr[3 + k]; }
    }
    TB_UNROLL1
    for (int o = 0; o < 3; o++) for (int s = S.ngl[o]; s < S.ncl[o]; s++) {
      const Con<sreal>& c = con_of(S, o, s);
      if (c.zone == ZONE_TOP) continue;
      sreal t[3];
      if (c.b2 == b) { cross3(t, c.r2, c.wr); for (int k = 0; k < 3; k++) { Fw[k] += c.wr[k]; Tw[k] += t[k] + c.wr[3 + k]; } }
      else if (c.b1 == b) { cross3(t, c.r1, c.wr); for (int k = 0; k < 3; k++) { Fw[k] -= c.wr[k]; Tw[k] -= t[k] + c.wr[3 + k]; } }
    }
    for (int k = 0; k < 3; k++) { N.fcon[k] = Fw[k]; N.fcon[3 + k] = Tw[k]; }
    sreal d[6], md[6];
    for (int k = 0; k < 6; k++) d[k] = B.warm[k] - N.asm_[k];
    mulM(m, b, N, d, md);
    for (int k = 0; k < 6; k++) {
      cpart += sreal(0.5) * md[k] * d[k];
      grad[k] = md[k] - N.fcon[k]; gn += grad[k] * grad[k];
    }
  }
  const sreal cost = sum3(cpart, base);
  gn = sum3(gn, base);
  return cost;
}

// Newton: Hessian.  Every bar lane builds its diagonal block from the contacts touching its bar, the owner of a
// bar-bar contact the block below the diagonal; all into shared memory
template <typename P>
TB_FN void newton_hessian(EnvSh<P>& S, const ModelT<typename P::real>& m, int b, const BarSolve<P>& N, int nmine, int ngr, bool bbmine, bool go) {
  typedef typename P::sreal sreal;
  if (!go) return;
  sreal H[21];
  for (int e = 0; e < 21; e++) H[e] = 0;
  H[0] = H[2] = H[5] = (sreal)m.M[6 * b];
  H[9] = N.Iw[0]; H[13] = N.Iw[1]; H[14] = N.Iw[2]; H[18] = N.Iw[3]; H[19] = N.Iw[4]; H[20] = N.Iw[5];
  S.cpl[b] = 0;
  TB_UNROLL1
  for (int s = 0; s < ngr; s++) {   // own ground contacts
    const Con<sreal>& c = con_of(S, b, s);
    if (c.zone == ZONE_TOP) continue;
    side_hessian(c, m, c.r2, H);
  }
  TB_UNROLL1
  for (int o = 0; o < 3; o++) for (int s = S.ngl[o]; s < S.ncl[o]; s++) {   // bar-bar contacts of all owners
    const Con<sreal>& c = con_of(S, o, s);
    if (c.zone == ZONE_TOP) continue;
    if (c.b2 != b && c.b1 != b) continue;
    side_hessian(c, m, c.b2 == b ? c.r2 : c.r1, H);
  }
  for (int e = 0; e < 21; e++) S.u.sol.D[b][e] = H[e];
  if (bbmine) {
    // this lane owns the pair p = b: rows = the higher bar, cols = the lower one
    sreal X[36];
    for (int e = 0; e < 36; e++) X[e] = 0;
    bool anyx = false;
    TB_UNROLL1
    for (int s = ngr; s < nmine; s++) {
      const Con<sreal>& c = con_of(S, b, s);
      if (c.zone == ZONE_TOP) continue;
      if (c.b2 > c.b1) cross_hessian(c, m, c.r2, c.r1, X); else cross_hessian(c, m, c.r1, c.r2, X);
      anyx = true;
    }
    if (anyx) { for (int e = 0; e < 36; e++) S.u.sol.O[b][e] = X[e]; S.cpl[b] = 1; }
  }
}

// Newton: search = H^-1 grad (the line search negates it).  Block LDL^T in the order bar 0, 1, 2, distributed by block row (lane b owns D[b]
// and the blocks left of it); absent blocks are skipped; fill-in can only appear in pair (2,1)
template <typename P> TB_FN void newton_solve(EnvSh<P>& S, int b, const typename P::sreal* grad, typename P::sreal* search, bool go) {
  typedef typename P::sreal sreal;
  const bool c10 = go && S.cpl[0] != 0, c20 = go && S.cpl[1] != 0, c21in = go && S.cpl[2] != 0;
  const bool f21 = c10 && c20, c21 = c21in || f21;
  sreal (*D)[21] = S.u.sol.D; sreal (*O)[36] = S.u.sol.O; sreal* dinv = S.u.sol.dinv; sreal* xs = S.u.sol.xv;
  const bool indep = go && (b == 0 || (b == 1 && !c10) || (b == 2 && !c20 && !c21));   // no block left of the diagonal
  const bool alone = indep && ((b == 0 && !c10 && !c20) || (b == 1 && !c21) || b == 2);   // and none below it
  sreal x[6];
  for (int k = 0; k < 6; k++) x[k] = grad[k];
  if (indep) { blk_ldl(D[b], dinv + 6 * b); blk_fwd(D[b], x); }
  if (alone) { for (int k = 0; k < 6; k++) x[k] *= dinv[6 * b + k]; blk_bwd(D[b], x); }
  if (any(go && (c10 || c20 || c21))) {
    if (go && b == 0 && !alone) for (int k = 0; k < 6; k++) xs[k] = x[k];   // z0
    wsync();
    // column 0: the off-diagonal blocks O10, O20 and the updates they cause, two rows per lane
    if (c10 || c20) {
      sreal Lr[21], dv[6];
      TB_UNROLL
      for (int e = 0; e < 21; e++) Lr[e] = D[0][e];
      TB_UNROLL
      for (int e = 0; e < 6; e++) dv[e] = dinv[e];
      if (c10) blk_trsm_rows2(O[0], Lr, dv, 2 * b);
      if (c20) blk_trsm_rows2(O[1], Lr, dv, 2 * b);
    }
    if (f21 && !c21in) for (int e = 0; e < 12; e++) O[2][12 * b + e] = 0;
    wsync();
    if (c10 || c20) {
      sreal d0[6], Bm[36];
      TB_UNROLL
      for (int k = 0; k < 6; k++) d0[k] = D[0][k * (k + 1) / 2 + k];
      if (c10) {
        TB_UNROLL
        for (int e = 0; e < 36; e++) Bm[e] = O[0][e];
        blk_mulsub_rows2(D[1], O[0], d0, Bm, true, 2 * b);
        if (f21) blk_mulsub_rows2(O[2], O[1], d0, Bm, false, 2 * b);
      }
      if (c20) {
        TB_UNROLL
        for (int e = 0; e < 36; e++) Bm[e] = O[1][e];
        blk_mulsub_rows2(D[2], O[1], d0, Bm, true, 2 * b);
      }
    }
    wsync();
    if (b == 1 && c10) {
      blk_ldl(D[1], dinv + 6);
      blk_gemv_sub(x, O[0], xs);
      blk_fwd(D[1], x);
    }
    if (go && b == 1 && !alone) for (int k = 0; k < 6; k++) xs[6 + k] = x[k];   // z1
    wsync();
    // column 1: O21 and its update of D2, two rows per lane
    if (c21) {
      sreal Lr[21], dv[6];
      TB_UNROLL
      for (int e = 0; e < 21; e++) Lr[e] = D[1][e];
      TB_UNROLL
      for (int e = 0; e < 6; e++) dv[e] = dinv[6 + e];
      blk_trsm_rows2(O[2], Lr, dv, 2 * b);
    }
    wsync();
    if (c21) {
      sreal d1[6], Bm[36];
      TB_UNROLL
      for (int k = 0; k < 6; k++) d1[k] = D[1][k * (k + 1) / 2 + k];
      TB_UNROLL
      for (int e = 0; e < 36; e++) Bm[e] = O[2][e];
      blk_mulsub_rows2(D[2], O[2], d1, Bm, true, 2 * b);
    }
    wsync();
    if (b == 2 && (c20 || c21)) {
      blk_ldl(D[2], dinv + 12);
      if (c20) blk_gemv_sub(x, O[1], xs);
      if (c21) blk_gemv_sub(x, O[2], xs + 6);
      blk_fwd(D[2], x);
      for (int k = 0; k < 6; k++) x[k] *= dinv[12 + k];
      blk_bwd(D[2], x);
      for (int k = 0; k < 6; k++) xs[12 + k] = x[k];   // final x2
    }
    wsync();
    if (go && b == 1 && !alone) {
      for (int k = 0; k < 6; k++) x[k] *= dinv[6 + k];
      if (c21) blk_gemvT_sub(x, O[2], xs + 12);
      blk_bwd(D[1], x);
      for (int k = 0; k < 6; k++) xs[6 + k] = x[k];   // final x1
    }
    wsync();
    if (go && b == 0 && !alone) {
      for (int k = 0; k < 6; k++) x[k] *= dinv[k];
      if (c10) blk_gemvT_sub(x, O[0], xs + 6);
      if (c20) blk_gemvT_sub(x, O[1], xs + 12);
      blk_bwd(D[0], x);
    }
  }
  if (go) for (int k = 0; k < 6; k++) search[k] = x[k];
}

// Newton: exact line search along the direction, which arrives as H^-1 grad in search and is negated here;
// mj_solPrimal's bracketing search as a per-env state machine.  Every tick evaluates cost / slope / curvature at ONE
// step size per env (3-lane sums), then each env advances its own bracketing logic, so the envs of a warp stay in lock
// step whatever their individual search sequences are.  cost: the env's cost at the iterate.  Returns the step size;
// evals: the cost evaluations it took
template <typename P>
TB_FN typename P::sreal line_search(const BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, const LaneCtx& L,
                                    const BarSolve<P>& N, const typename P::sreal* grad, typename P::sreal* search, int nmine,
                                    bool go, typename P::sreal cost, int& evals) {
  typedef typename P::sreal sreal;
  const int b = L.bar, base = L.base;
  const sreal SMINV = Lim<sreal>::MINVAL;
  // the negation sits here, next to its uses, so that the compiler folds it into the sums below (mul + sub) instead of
  // contracting them into FMAs: the rounding of gs, qG1 and qG2 depends on it
  if (go) for (int k = 0; k < 6; k++) search[k] = -search[k];
  sreal snorm = 0, gs = 0, qG1 = 0, qG2 = 0, gauss = 0;
  if (go) {
    sreal d[6], md[6], ms[6];
    for (int k = 0; k < 6; k++) d[k] = B.warm[k] - N.asm_[k];
    mulM(m, b, N, d, md); mulM(m, b, N, search, ms);
    for (int k = 0; k < 6; k++) {
      sreal sk = search[k];
      snorm += sk * sk; gs += grad[k] * sk;
      qG1 += sk * md[k];
      qG2 += sreal(0.5) * sk * ms[k];
      gauss += sreal(0.5) * md[k] * d[k];
    }
  }
  snorm = sum3(snorm, base); gs = sum3(gs, base);
  snorm = tsqrt(snorm);
  wsync();
  publish(S, b, search, go);
  wsync();
  if (go && nmine > 0) {
    TB_UNROLL1
    for (int s = 0; s < nmine; s++) {
      Con<sreal>& k = con_of(S, b, s);
      con_mulJ(k, S.u.sol.xv, k.jv);
      sreal q0 = 0, q1 = 0, q2 = 0, UU = 0, UV = 0, VV = 0;
      for (int j = 0; j < 6; j++) {
        sreal D = k.D0 * (sreal)m.dscale[j], ja = k.jar[j], jv = k.jv[j];
        q0 += sreal(0.5) * D * ja * ja; q1 += D * ja * jv; q2 += sreal(0.5) * D * jv * jv;
        if (j > 0) { sreal U = ja * (sreal)m.fr[j - 1], V = jv * (sreal)m.fr[j - 1]; UU += U * U; UV += U * V; VV += V * V; }
      }
      k.t.ls.q0 = q0; k.t.ls.q1 = q1; k.t.ls.q2 = q2;
      k.t.ls.U0 = k.jar[0] * (sreal)m.mu; k.t.ls.V0 = k.jv[0] * (sreal)m.mu; k.t.ls.UU = UU; k.t.ls.UV = UV; k.t.ls.VV = VV;
    }
  }
  sreal alpha = 0;
  evals = 1;
  LsCoef<sreal> lc0 = LsCoef<sreal>();   // the lane's first contact stays in registers for the evaluations
  if (go && nmine > 0) lc0 = ls_coef(con_of(S, b, 0));
  struct Pnt { sreal alpha, cost, d0, d1; };
  // W_*: waiting for the evaluation it requested; L_*: pure logic, resolved without an evaluation
  enum { W_P1 = 0, W_A, W_P1NEXT, W_MID, W_B1, W_B2, L_ACHECK, L_AFTERA, L_BCHECK, L_DOB2, L_ENDITER, L_FINAL, LS_DONE };
  const sreal gtol = (sreal)m.tol * (sreal)m.ls_tol * snorm * ((sreal)m.meaninertia * NV);
  const int maxe = m.ls_iterations;
  Pnt p0, p1, p2, pmid, p1next, p2next, c0;
  p0.alpha = 0; p0.cost = cost; p0.d0 = gs; p0.d1 = -gs > 0 ? -gs : SMINV;   // alpha = 0 is analytic (H search = -grad)
  p1 = p2 = pmid = p1next = p2next = c0 = p0;
  int st = LS_DONE, dirn = 1;
  bool p2update = false, b1 = false, b2 = false;
  sreal aeval = 0;
  auto newton = [&](const Pnt& p) { return p.alpha - tdiv(p.d0, p.d1); };
  // update_bracket against the candidates captured at the mid-point evaluation: (old p1next = c0, p2next, pmid)
  auto bracket1 = [&](Pnt& p, const Pnt& q, int& flag) {
    if (p.d0 < 0 && q.d0 < 0 && p.d0 < q.d0) { p = q; flag = 1; }
    else if (p.d0 > 0 && q.d0 > 0 && p.d0 > q.d0) { p = q; flag = 2; }
  };
  auto bracket = [&](Pnt& p) {
    int flag = 0;
    bracket1(p, c0, flag); bracket1(p, p2next, flag); bracket1(p, pmid, flag);
    return flag;
  };
  if (go && !(snorm < SMINV)) { st = W_P1; aeval = newton(p0); }
  TB_UNROLL1
  for (;;) {
    const bool ev = st != LS_DONE;
    if (!any(ev)) break;
    sreal c_ = 0, d0_ = 0, d1_ = 0;
    if (ev) {
      if (nmine > 0) {
        con_ls(lc0, m, aeval, c_, d0_, d1_);
        TB_UNROLL1
        for (int s = 1; s < nmine; s++) con_ls(ls_coef(con_of(S, b, s)), m, aeval, c_, d0_, d1_);
      }
      c_ += aeval * aeval * qG2 + aeval * qG1 + gauss; d0_ += 2 * aeval * qG2 + qG1; d1_ += 2 * qG2;
    }
    Pnt r;
    r.alpha = aeval; r.cost = sum3(c_, base); r.d0 = sum3(d0_, base); r.d1 = sum3(d1_, base);
    if (r.d1 <= 0) r.d1 = SMINV;
    if (ev) {
      evals++;
      switch (st) {
        case W_P1:
          p1 = r;
          if (p0.cost < p1.cost) p1 = p0;
          if (tabs(p1.d0) < gtol) { alpha = p1.alpha; st = LS_DONE; }
          else { dirn = p1.d0 < 0 ? 1 : -1; p2 = p1; p2update = false; st = L_ACHECK; }
          break;
        case W_A:
          p1 = r;
          if (tabs(p1.d0) < gtol) { alpha = p1.alpha; st = LS_DONE; } else st = L_ACHECK;
          break;
        case W_P1NEXT: p1next = r; st = L_BCHECK; break;
        case W_MID: {
          pmid = r;
          c0 = p1next;
          int best = -1; sreal bestcost = 0, bestalpha = 0;
          if (tabs(c0.d0) < gtol) { bestcost = c0.cost; bestalpha = c0.alpha; best = 0; }
          if (tabs(p2next.d0) < gtol && (best == -1 || p2next.cost < bestcost)) { bestcost = p2next.cost; bestalpha = p2next.alpha; best = 1; }
          if (tabs(pmid.d0) < gtol && (best == -1 || pmid.cost < bestcost)) { bestcost = pmid.cost; bestalpha = pmid.alpha; best = 2; }
          if (best >= 0) { alpha = bestalpha; st = LS_DONE; }
          else {
            b1 = bracket(p1) != 0;
            if (b1) { aeval = newton(p1); st = W_B1; } else st = L_DOB2;
          }
          break;
        }
        case W_B1: p1next = r; st = L_DOB2; break;
        case W_B2: p2next = r; st = L_ENDITER; break;
        default: break;
      }
      TB_UNROLL1
      for (;;) {   // logic transitions until the env requests an evaluation or finishes
        if (st == L_ACHECK) {
          if (p1.d0 * dirn <= -gtol && evals < maxe) { p2 = p1; p2update = true; aeval = newton(p1); st = W_A; }
          else st = L_AFTERA;
        } else if (st == L_AFTERA) {
          if (evals >= maxe || !p2update) { alpha = p1.alpha; st = LS_DONE; }
          else { p2next = p1; aeval = newton(p1); st = W_P1NEXT; }
        } else if (st == L_BCHECK) {
          if (evals < maxe) { aeval = sreal(0.5) * (p1.alpha + p2.alpha); st = W_MID; } else st = L_FINAL;
        } else if (st == L_DOB2) {
          b2 = bracket(p2) != 0;
          if (b2) { aeval = newton(p2); st = W_B2; } else st = L_ENDITER;
        } else if (st == L_ENDITER) {
          if (!b1 && !b2) { alpha = pmid.alpha; st = LS_DONE; } else st = L_BCHECK;
        } else if (st == L_FINAL) {
          if (p1.cost <= p2.cost && p1.cost < p0.cost) alpha = p1.alpha;
          else if (p2.cost <= p1.cost && p2.cost < p0.cost) alpha = p2.alpha;
          else alpha = 0;
          st = LS_DONE;
        } else break;
      }
    }
  }
  return alpha;
}

// Newton: move the iterate and the rows of this lane's contacts by alpha along the search direction
template <typename P>
TB_FN void newton_move(BarState<P>& B, EnvSh<P>& S, int b, const typename P::sreal* search, int nmine, typename P::sreal alpha) {
  typedef typename P::sreal sreal;
  for (int k = 0; k < 6; k++) B.warm[k] += alpha * search[k];
  if (nmine > 0) {
    TB_UNROLL1
    for (int s = 0; s < nmine; s++) {
      Con<sreal>& c = con_of(S, b, s);
      for (int r = 0; r < 6; r++) c.jar[r] += alpha * c.jv[r];
    }
  }
}

// implicitfast + advance: (M - h D) x = qfrc_smooth + qfrc_constraint on the bar's 6x6 block (Cholesky, packed
// lower), then velocity, position and orientation
template <typename P>
TB_FN void implicitfast(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, int b, const BarFrame<P>& F,
                        const BarSolve<P>& N, const typename P::real* Dblk) {
  typedef typename P::real real; typedef typename P::sreal sreal;
  const real h = m.h;
  const real* Mb = m.M + 6 * b;
  real A[21], x[6];
  for (int e = 0; e < 21; e++) A[e] = -h * Dblk[e];
  {
    sreal al[3], fl[3];
    mulMTV(al, F.Rs, N.asm_ + 3); mulMTV(fl, F.Rs, N.fcon + 3);   // qacc_smooth and the constraint torque in body coordinates
    for (int r = 0; r < 3; r++) { x[r] = (real)((sreal)Mb[r] * N.asm_[r] + N.fcon[r]); x[3 + r] = (real)((sreal)Mb[3 + r] * al[r] + fl[r]); }
  }
  for (int r = 0; r < 6; r++) A[r * (r + 1) / 2 + r] += Mb[r];
  TB_UNROLL
  for (int j = 0; j < 6; j++) {
    real s = A[j * (j + 1) / 2 + j];
    TB_UNROLL
    for (int k = 0; k < j; k++) s -= A[j * (j + 1) / 2 + k] * A[j * (j + 1) / 2 + k];
    real inv = trcp(tsqrt(s));
    A[j * (j + 1) / 2 + j] = inv;   // 1 / L_jj
    TB_UNROLL
    for (int i = j + 1; i < 6; i++) {
      real t = A[i * (i + 1) / 2 + j];
      TB_UNROLL
      for (int k = 0; k < j; k++) t -= A[i * (i + 1) / 2 + k] * A[j * (j + 1) / 2 + k];
      A[i * (i + 1) / 2 + j] = t * inv;
    }
  }
  TB_UNROLL
  for (int i = 0; i < 6; i++) {
    real t = x[i];
    TB_UNROLL
    for (int k = 0; k < i; k++) t -= A[i * (i + 1) / 2 + k] * x[k];
    x[i] = t * A[i * (i + 1) / 2 + i];
  }
  TB_UNROLL
  for (int i = 5; i >= 0; i--) {
    real t = x[i];
    TB_UNROLL
    for (int k = i + 1; k < 6; k++) t -= A[k * (k + 1) / 2 + i] * x[k];
    x[i] = t * A[i * (i + 1) / 2 + i];
  }
  for (int k = 0; k < 6; k++) B.v[k] += h * x[k];
  for (int k = 0; k < 3; k++) B.x[k] += h * B.v[k];
  real ax[3] = {B.v[3], B.v[4], B.v[5]}, qr[4], qn[4];
  real ang = h * normalize3(ax);
  if (ang == 0) { qr[0] = 1; qr[1] = qr[2] = qr[3] = 0; }
  else { real sn, cs; tsincos(ang * real(0.5), &sn, &cs); qr[0] = cs; qr[1] = ax[0] * sn; qr[2] = ax[1] * sn; qr[3] = ax[2] * sn; }
  normalize4(B.q);
  const real* a = B.q;
  qn[0] = a[0] * qr[0] - a[1] * qr[1] - a[2] * qr[2] - a[3] * qr[3];
  qn[1] = a[0] * qr[1] + a[1] * qr[0] + a[2] * qr[3] - a[3] * qr[2];
  qn[2] = a[0] * qr[2] - a[1] * qr[3] + a[2] * qr[0] + a[3] * qr[1];
  qn[3] = a[0] * qr[3] + a[1] * qr[2] - a[2] * qr[1] + a[3] * qr[0];
  for (int k = 0; k < 4; k++) B.q[k] = qn[k];
  if (m.dyntype && b == 0) for (int i = 0; i < NACT; i++) S.act[i] += (double)(h * S.actdot[i]);
}

// ------------------------------------------------------------------ one physics pass
// mj_forward (integ = false) or mj_step (integ = true) for the envs of the warp that are `on`.  The bar state B is
// the lane's registers; the env's contacts of the last pass stay in S on return.  This driver holds every CTA barrier
// of the pass (uni_any with `aligned`): the loop heads of the Newton iteration and of the mj_checkAcc retry.
template <typename P>
TB_FN void phys(BarState<P>& B, EnvSh<P>& S, const ModelT<typename P::real>& m, const LaneCtx& L, bool on, bool integ, bool aligned) {
  typedef typename P::sreal sreal;
  const int b = L.bar, base = L.base;
  if (integ) check_state(B, S, m, L, on);
  BarFrame<P> F;
  BarSolve<P> N;
  typename P::real Dblk[21];
  bool pass_on = on;
  TB_UNROLL1
  for (int pass = 0; pass < 2; pass++) {
    kinematics(B, S, m, b, F, pass_on);
    wsync();
    smooth_dynamics(B, S, m, b, F, N, Dblk, pass_on);
    wsync();   // the tendon end points are dead: their storage now carries the solver's exchange
    publish(S, b, N.asm_, pass_on);
    int nmine = 0, nmpr = 0;
    if (m.floor_type == 0) collide_plane(B, S, m, b, F, nmine, pass_on);
    else collide_hfield(B, S, m, b, F, nmine, nmpr, pass_on);
    const int ngr = nmine;   // ground contacts come first in the lane's list
    collide_bars(S, m, b, nmine, nmpr, pass_on);
    if (pass_on) { S.ncl[b] = nmine; S.ngl[b] = ngr; }
    wsync();
    bool bbmine;
    const sreal csm = contact_rows(S, m, b, nmine, pass_on, bbmine);
    const int nact_env = isum3(pass_on ? nmine : 0, base);
    {
      int nm = isum3(pass_on ? nmpr : 0, base);
      if (pass_on && b == 0) { S.nact = nact_env; S.nmpr += nm; }
    }
    // ---------------- mj_fwdConstraint: warm-start choice + Newton
    bool act = pass_on && nact_env > 0;
    warm_start(B, S, m, L, N, nmine, csm, act, pass_on);
    for (int k = 0; k < 6; k++) N.fcon[k] = 0;
    sreal grad[6], search[6] = {0, 0, 0, 0, 0, 0};
    sreal cost = 0, oldcost = 0;
    int iter = 0, nls = 0;
    bool first = true;
    TB_UNROLL1
    for (;;) {
      if (!uni_any(act, aligned)) break;
      sreal gn;
      const sreal newcost = newton_gradient(B, S, m, L, N, nmine, ngr, act, grad, gn);
      if (act) {
        oldcost = cost; cost = newcost;
        if (!first && ((sreal)m.solscale * (oldcost - cost) < (sreal)m.tol || gn < (sreal)m.gradtol * (sreal)m.gradtol)) act = false;   // converged
      }
      first = false;
      const bool go = act && iter < m.iterations;
      if (!go) act = false;
      if (!any(go)) {
        // an aligned warp goes back to the CTA barrier at the loop head, and keeps meeting it until every warp of the
        // CTA has converged
        if (aligned) continue;
        break;
      }
      newton_hessian(S, m, b, N, nmine, ngr, bbmine, go);
      wsync();
      newton_solve(S, b, grad, search, go);
      int evals;
      const sreal alpha = line_search(B, S, m, L, N, grad, search, nmine, go, cost, evals);
      if (go) {
        nls += evals;
        if (alpha == 0) act = false;
        else { newton_move(B, S, b, search, nmine, alpha); iter++; }
      }
      wsync();
    }
    if (pass_on) {   // the iterate back to body coordinates: it is the next warm start
      sreal wl[3];
      mulMTV(wl, F.Rs, B.warm + 3);
      for (int k = 0; k < 3; k++) B.warm[3 + k] = wl[k];
      if (nact_env > 0 && b == 0) { S.niter += iter; S.nls += nls; }
    }
    // ---------------- mj_checkAcc: a bad acceleration resets the env and repeats the forward pass
    if (!integ || pass == 1) break;
    bool bad = false;
    for (int k = 0; k < 6; k++) bad |= is_bad(B.warm[k]);
    bad = grp_any(bad && on, base);
    if (!uni_any(bad, aligned)) break;
    pass_on = on && bad;
    if (pass_on) { if (b == 0) S.bad |= 4; reset_bar(B, S, m, b); }
    wsync();
  }
  if (integ && on) implicitfast(B, S, m, b, F, N, Dblk);
  wsync();
}

// mj_rnePostConstraint: cfrc_ext rows [torque; force] for world + 3 bars about the (stale) body positions, from the
// contacts of the last pass; also the total bar-bar contact force magnitude (run.py:155-161).  Leaves S.cfrc.
template <typename P>
TB_FN void cfrc_stage(EnvSh<P>& S, const ModelT<typename P::real>& m, const LaneCtx& L, bool on) {
  typedef typename P::real real;
  typedef typename P::sreal sreal;
  const int b = L.bar, base = L.base;
  sreal own[6] = {0, 0, 0, 0, 0, 0}, world[6] = {0, 0, 0, 0, 0, 0}, barf = 0;
  if (on && S.nact > 0) {
    // the world row is taken about the mass-weighted centre of the three bars
    sreal com[3] = {0, 0, 0}, mt = 0;
    for (int bb = 0; bb < NBAR; bb++) { for (int k = 0; k < 3; k++) com[k] += (sreal)S.xpos[3 * bb + k] * (sreal)m.M[6 * bb]; mt += (sreal)m.M[6 * bb]; }
    scl3(com, com, 1 / mt);
    for (int o = 0; o < 3; o++) for (int s = 0; s < S.ncl[o]; s++) {
      const Con<sreal>& c = con_of(S, o, s);
      if (c.zone == ZONE_TOP) continue;
      sreal t[3];
      if (c.b2 == b) {
        cross3(t, c.r2, c.wr);
        for (int k = 0; k < 3; k++) { own[k] += t[k] + c.wr[3 + k]; own[3 + k] += c.wr[k]; }
        if (c.b1 < 0) {
          sreal r[3];
          for (int k = 0; k < 3; k++) r[k] = (sreal)S.xpos[3 * b + k] + c.r2[k] - com[k];
          cross3(t, r, c.wr);
          for (int k = 0; k < 3; k++) { world[k] -= t[k] + c.wr[3 + k]; world[3 + k] -= c.wr[k]; }
        }
      } else if (c.b1 == b) {
        cross3(t, c.r1, c.wr);
        for (int k = 0; k < 3; k++) { own[k] -= t[k] + c.wr[3 + k]; own[3 + k] -= c.wr[k]; }
      }
      if (c.b1 >= 0 && c.owner == b) barf += tsqrt(c.wr[0] * c.wr[0] + c.wr[1] * c.wr[1] + c.wr[2] * c.wr[2]);
    }
  }
  for (int k = 0; k < 6; k++) world[k] = sum3(world[k], base);
  barf = sum3(barf, base);
  if (on) {
    for (int k = 0; k < 6; k++) S.cfrc[6 * (b + 1) + k] = (real)own[k];
    if (b == 0) { for (int k = 0; k < 6; k++) S.cfrc[k] = (real)world[k]; S.barforce = barf; }
  }
  wsync();
}

}  // namespace tb
