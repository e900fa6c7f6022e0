// tb_env.cuh -- tr_env / tensegrity_env semantics around the bar-lane physics.
//   step    : tr_env.py:327-527 ; tensegrity_env.py:291-410
//   obs     : tr_env.py:529-646 ; tensegrity_env.py:412-430
//   reset   : tr_env.py:709-872 ; tensegrity_env.py:433-512  (+ gym MujocoEnv.reset / set_state)
// The env-level arithmetic (pose, reward, termination, observation: a few hundred scalar operations per env step,
// always fp64) is done by lane 0 of the env's three lanes; the physics calls in between are warp-collective
// (simulate()), so every routine here that contains one is entered by all 32 lanes with a per-env `on` predicate.
#pragma once
#include "tb_core.cuh"

namespace tb {

struct Aux {  // env bookkeeping (valid in lane 0 of the env)
  double xy_prev[2], psi_prev, reset_psi, waypt[2], ori[2];
  double step_num, ep_ret, ep_len, xvel, yvel;
  int head_n, head_pos;
  double* heading;  // [HEADING_SLOTS] in global memory
  const double* draws;  // [NDRAW] in global memory: the random draws of the env's current reset
  unsigned long long nz_seed, nz_stream, nz_nreset;   // keys of the reset-noise draws
};
struct StepOut {
  double reward, fwd, ctrl_cost, info_ctrl, healthy, psi, xy[2];   // info_ctrl: what info["reward_ctrl"] reports
  int terminated;
  double maxcfrc, barforce;
};
struct Pose { double xy[2], left[3], right[3], psi; };

struct StepIO {
  double* state;        // [N + n_pool][STATE_STRIDE]
  double* heading;      // [N + n_pool][HEADING_SLOTS]
  const double* ctrl64; // [N][6] or null
  const float* ctrl32;  // [N][6] or null
  double* obs;          // [N][obs_dim] or null
  float* obs32;         // [N][obs_dim] or null
  double* reward;       // [N] or null
  uint8_t* done;        // [N] or null (terminated | truncated)
  double* info;         // [N][INFO_DIM] or null
  double* term_obs;     // [N][obs_dim] or null : observation before an auto reset
  double* draws;        // [N + n_pool][NDRAW]: reset draws (in: explicit, out: generated)
  const uint8_t* mask;  // reset: which envs ; null = all
  unsigned long long seed;
  long long env_id_base;
  int n_envs;
  int explicit_draws;
  int n_pool;           // background reset pool slots stored after the n_envs records
  double* pool_obs;     // [n_pool][obs_dim]: reset observation of each ready pool slot
  double* pool_real_obs;// [n_pool][obs_dim] or null: its noise-free twin (use_obs_noise)
  double* real_obs;     // [N][obs_dim] or null: noise-free observation when use_obs_noise (info["real_observation"])
  int* counter;         // work counter of the launch
  double* params;       // per-env variant: [N + n_pool][NPARAM] parameter rows
  const double* prange; // per-env variant: {nominal, lo, hi}[NPARAM] of the reset draws, or null = rows kept at resets
};

TB_FN double angle_normalize(double t) {  // tr_env.py:648-654
  while (t > PI) t -= 2 * PI;
  while (t <= -PI) t += 2 * PI;
  return t;
}
// COM / left-right end-cap centroids from the (stale) kinematics of the last forward pass
template <typename PR> TB_FN void read_pose(const EnvSh<PR>& S, Pose& P) {
  P.xy[0] = ((double)S.xpos[0] + (double)S.xpos[3] + (double)S.xpos[6]) / 3;
  P.xy[1] = ((double)S.xpos[1] + (double)S.xpos[4] + (double)S.xpos[7]) / 3;
  for (int k = 0; k < 3; k++) {
    P.left[k] = ((double)S.sph[3 * 0 + k] + (double)S.sph[3 * 2 + k] + (double)S.sph[3 * 4 + k]) / 3;   // s0, s2, s4
    P.right[k] = ((double)S.sph[3 * 1 + k] + (double)S.sph[3 * 3 + k] + (double)S.sph[3 * 5 + k]) / 3;  // s1, s3, s5
  }
  P.psi = atan2(-(P.left[0] - P.right[0]), P.left[1] - P.right[1]);
}
TB_FN double ditch_reward(const EnvCfg& c, const Aux& A, const double* xy) {  // tr_env.py:656-667
  double pv[2] = {A.waypt[0] - A.ori[0], A.waypt[1] - A.ori[1]};
  double dp = sqrt(pv[0] * pv[0] + pv[1] * pv[1]);
  double pn[2] = {pv[0] / dp, pv[1] / dp};
  double tv[2] = {A.waypt[0] - xy[0], A.waypt[1] - xy[1]};
  double along = tv[0] * pn[0] + tv[1] * pn[1];
  double bx = tv[0] - along * pn[0], by = tv[1] - along * pn[1];
  double bias = sqrt(bx * bx + by * by);
  double ditch = c.ditch_reward_max * (1.0 - fabs(along) / dp) * exp(-(bias * bias) / (2 * c.ditch_reward_stdev * c.ditch_reward_stdev));
  double dx = xy[0] - A.waypt[0], dy = xy[1] - A.waypt[1];
  double dn = sqrt(dx * dx + dy * dy);
  double wp = c.waypt_reward_amplitude * exp(-(dn * dn) / (2 * c.waypt_reward_stdev * c.waypt_reward_stdev));
  return ditch + wp;
}
// scipy Rotation.from_matrix(M).as_quat() -> (x, y, z, w)
TB_FN void mat2quat_scipy(const double* M, double* q) {
  double tr = M[0] + M[4] + M[8];
  double dec[4] = {M[0], M[4], M[8], tr};
  int ch = 0;
  for (int i = 1; i < 4; i++) if (dec[i] > dec[ch]) ch = i;
  if (ch != 3) {
    int i = ch, j = (i + 1) % 3, k = (j + 1) % 3;
    q[i] = 1 - tr + 2 * M[4 * i];
    q[j] = M[3 * j + i] + M[3 * i + j];
    q[k] = M[3 * k + i] + M[3 * i + k];
    q[3] = M[3 * k + j] - M[3 * j + k];
  } else {
    q[0] = M[7] - M[5]; q[1] = M[2] - M[6]; q[2] = M[3] - M[1]; q[3] = 1 + tr;
  }
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int i = 0; i < 4; i++) q[i] /= n;
}
// Philox4x32-10, counter = (env id, reset count), key = seed
TB_FN void philox(unsigned long long seed, unsigned long long ctr_lo, unsigned long long ctr_hi, uint32_t out[4]) {
  uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32), c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; r++) {
    unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
TB_FN double u01(uint32_t a, uint32_t b) {  // 53-bit uniform in [0,1)
  unsigned long long x = (((unsigned long long)a << 32) | b) >> 11;
  return (double)x * (1.0 / 9007199254740992.0);
}
// reset noise (tr_env.py:734-743): component i of the 21 uniform qpos offsets (i < 21) / 18 normal qvel values, unscaled
TB_FN double reset_noise_draw(unsigned long long seed, unsigned long long stream, unsigned long long nreset, int i) {
  uint32_t r[4];
  philox(seed ^ 0x72657365746e7365ull, stream, (nreset << 8) | (unsigned long long)i, r);
  if (i < NQ) return 2.0 * u01(r[0], r[1]) - 1.0;
  double u1 = 1.0 - u01(r[0], r[1]), u2 = u01(r[2], r[3]);
  return sqrt(-2.0 * log(u1)) * cos(2 * PI * u2);
}
// the pr-th pair of standard normals of one observation (Philox + Box-Muller)
TB_FN void noise_pair(unsigned long long seed, unsigned long long stream, unsigned long long nreset,
                      unsigned long long step, int pr, double& z0, double& z1) {
  uint32_t r[4];
  philox(seed ^ 0x6f62736e6f697365ull, stream, (((nreset << 24) | (step & 0xffffffull)) << 8) | (unsigned long long)pr, r);
  double u1 = 1.0 - u01(r[0], r[1]), u2 = u01(r[2], r[3]);
  double rad = sqrt(-2.0 * log(u1));
  z0 = rad * cos(2 * PI * u2); z1 = rad * sin(2 * PI * u2);
}
// Observation noise (tr_env.py:552-644): every component of the cap positions / cap velocities gets
// N(0, obs_noise_cap_pos_stdev), every tendon length N(0, obs_noise_tendon_stdev); the tracking vector loses the mean
// cap-position noise and the target yaw is re-derived from it (:626-639); the vel_track command passes (:641-644).
TB_NOINL void obs_noise(const EnvCfg& c, double* obs, unsigned long long seed, unsigned long long stream,
                        unsigned long long nreset, unsigned long long step) {
  const int nvel = c.use_cap_velocity ? 18 : 0, n = 27 + nvel;
  const double sp = c.obs_noise_cap_pos_stdev, st = c.obs_noise_tendon_stdev;
  double cn0 = 0, cn1 = 0;   // mean of the noisy centroid-relative cap positions (x, y)
  for (int pr = 0; pr < (n + 1) / 2; pr++) {
    double z[2];
    noise_pair(seed, stream, nreset, step, pr, z[0], z[1]);
    for (int h = 0; h < 2; h++) {
      int i = 2 * pr + h;
      if (i >= n) break;
      obs[i] = (i < 18 + nvel ? sp : st) * z[h] + obs[i];
      if (i < 18 && i % 3 == 0) cn0 += obs[i];
      if (i < 18 && i % 3 == 1) cn1 += obs[i];
    }
  }
  cn0 /= 6; cn1 /= 6;
  if (c.task == TASK_TRACKING || c.task == TASK_AIMING) {
    double tx = obs[n] - cn0, ty = obs[n + 1] - cn1, nn = sqrt(tx * tx + ty * ty);
    obs[n] = tx; obs[n + 1] = ty; obs[n + 2] = atan2(ty / nn, tx / nn);
  }
}

// observation (stale positions / tendon lengths, fresh qvel) -- lane 0
template <typename PR>
TB_NOINL void compute_obs(const EnvSh<PR>& S, const EnvCfg& c, const Aux& A, double* obs) {
  if (c.env_kind == ENV_LEGACY) {
    for (int b = 0; b < 3; b++) {  // geom rXY: body frame with x, y columns negated (geom quat 0 0 0 1)
      double R[9];
      for (int k = 0; k < 9; k++) R[k] = (double)S.xmat[9 * b + k];
      double Gm[9] = {-R[0], -R[1], R[2], -R[3], -R[4], R[5], -R[6], -R[7], R[8]};
      mat2quat_scipy(Gm, obs + 4 * b);
    }
    for (int i = 0; i < 18; i++) obs[12 + i] = S.u.home.qvel[i];
    for (int i = 0; i < 9; i++) obs[30 + i] = (double)S.tlen[i];
    return;
  }
  double cen[3] = {0, 0, 0};
  for (int b = 0; b < NBAR; b++)
    for (int k = 0; k < 3; k++) cen[k] += (double)S.sph[3 * (2 * b) + k] + (double)S.sph[3 * (2 * b + 1) + k];
  for (int k = 0; k < 3; k++) cen[k] /= 6;
  int nvel = c.use_cap_velocity ? 18 : 0;
  for (int i = 0; i < 18; i++) obs[i] = (double)S.sph[i] - cen[i % 3];
  if (nvel) for (int cap = 0; cap < 6; cap++) {
    int b = cap / 2;
    double r[3], w[3] = {S.u.home.qvel[6 * b + 3], S.u.home.qvel[6 * b + 4], S.u.home.qvel[6 * b + 5]}, cr[3];
    for (int k = 0; k < 3; k++) r[k] = (double)S.sph[3 * cap + k] - (double)S.xpos[3 * b + k];
    cross3(cr, w, r);  // local-frame angular velocity used as if world-frame (tr_env.py:599-604)
    for (int k = 0; k < 3; k++) obs[18 + 3 * cap + k] = S.u.home.qvel[6 * b + k] + cr[k];
  }
  for (int i = 0; i < 9; i++) obs[18 + nvel + i] = (double)S.tlen[i];
  int base = 27 + nvel;
  if (c.task == TASK_TRACKING || c.task == TASK_AIMING) {
    double tx = A.waypt[0] - cen[0], ty = A.waypt[1] - cen[1], n = sqrt(tx * tx + ty * ty);
    obs[base] = tx; obs[base + 1] = ty; obs[base + 2] = atan2(ty / n, tx / n);
  } else if (c.task == TASK_VEL_TRACK) {
    obs[base] = 0.5 * cos(A.reset_psi); obs[base + 1] = 0.5 * sin(A.reset_psi); obs[base + 2] = 0.0;
  }
}

// do_simulation(ctrl, nsub) (integ) or mj_forward (integ = false, nsub = 1) on the env state in S, then
// mj_rnePostConstraint.  Warp-collective.  The bar state is register-resident for the whole call.
template <typename PR>
TB_NOINL void simulate(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const LaneCtx& L, bool on, int nsub, bool integ, bool aligned) {
  typedef typename PR::real real;
  typedef typename PR::sreal sreal;
  BarState<PR> B;
  const int b = L.bar;
  for (int k = 0; k < 3; k++) B.x[k] = (real)S.u.home.qpos[7 * b + k];
  for (int k = 0; k < 4; k++) B.q[k] = (real)S.u.home.qpos[7 * b + 3 + k];
  for (int k = 0; k < 6; k++) { B.v[k] = (real)S.u.home.qvel[6 * b + k]; B.warm[k] = (sreal)S.u.home.warm[6 * b + k]; }
  wsync();
  TB_UNROLL1
  for (int s = 0; s < nsub; s++) {
    if (aligned) uni_any(true, true);   // the warps of the CTA enter every substep together
    phys(B, S, m, L, on, integ, aligned);
  }
  cfrc_stage(S, m, L, on);
  wsync();
  if (on) {
    for (int k = 0; k < 3; k++) S.u.home.qpos[7 * b + k] = (double)B.x[k];
    for (int k = 0; k < 4; k++) S.u.home.qpos[7 * b + 3 + k] = (double)B.q[k];
    for (int k = 0; k < 6; k++) { S.u.home.qvel[6 * b + k] = (double)B.v[k]; S.u.home.warm[6 * b + k] = (double)B.warm[k]; }
  }
  wsync();
}

// heading ring buffer (the reference's deque, never cleared across episodes) lives in global memory -- lane 0
TB_FN void heading_push(Aux& A, double v) { A.heading[(A.head_pos + A.head_n) % HEADING_SLOTS] = v; A.head_n++; }
TB_FN double heading_pop(Aux& A) {
  double v = A.heading[A.head_pos];
  A.head_pos = (A.head_pos + 1) % HEADING_SLOTS;
  A.head_n--;
  return v;
}

// the part of env.step after do_simulation -- lane 0
template <typename PR>
TB_NOINL void env_step_post(EnvSh<PR>& S, const EnvCfg& c, Aux& A, StepOut& O) {
  const double dt = c.dt;
  double xy_before[2] = {A.xy_prev[0], A.xy_prev[1]}, psi_before = A.psi_prev;
  Pose P; read_pose(S, P);
  double xvel = (P.xy[0] - xy_before[0]) / dt, yvel = (P.xy[1] - xy_before[1]) / dt;
  A.xvel = xvel; A.yvel = yvel;
  double psi_after = P.psi;
  if (c.env_kind == ENV_LEGACY && c.task == TASK_TURN)  // tensegrity_env.py:320-322
    psi_after = atan2(P.right[1] - P.left[1], P.right[0] - P.left[0]);
  double psi_info = psi_after;
  double cc = 0;
  for (int i = 0; i < NACT; i++) {
    double a = S.action[i];
    double v = (c.env_kind == ENV_TR) ? (a + 0.5 - (double)S.tlen[i]) : a;
    cc += v * v;
  }
  cc *= c.ctrl_cost_weight;
  double fwd = 0, ctrl_cost = cc;
  double healthy = c.terminate_when_unhealthy ? c.healthy_reward : 0.0;
  int delay = c.reward_delay_steps;
  bool finite = true;
  for (int i = 0; i < NQ; i++) finite &= isfinite(S.u.home.qpos[i]);
  for (int i = 0; i < NV; i++) finite &= isfinite(S.u.home.qvel[i]);
  bool moving_any = false;
  for (int i = 0; i < NV; i++) moving_any |= fabs(S.u.home.qvel[i]) > 0.1;
  bool healthy_turn = finite && moving_any;
  bool healthy_lin = finite && ((xvel > 1e-4 || xvel < -1e-4) || (yvel > 1e-4 || yvel < -1e-4));
  bool is_healthy = healthy_lin;
  bool extra_term = false;
  if (c.task == TASK_TURN) {
    is_healthy = healthy_turn;
    heading_push(A, psi_after);
    if (A.head_n > delay) {
      double old_psi = heading_pop(A), pa = psi_after;
      if (pa < -PI / 2 && old_psi > PI / 2) pa = 2 * PI + pa;
      else if (pa > PI / 2 && old_psi < -PI / 2) pa = -2 * PI + pa;
      psi_info = pa;
      fwd = (pa - old_psi) / (dt * delay) * c.desired_direction;
    } else { fwd = 0; ctrl_cost = 0; }
  } else if (c.task == TASK_STRAIGHT) {
    double dx = P.xy[0] - xy_before[0], dy = P.xy[1] - xy_before[1];
    double psi_diff = fabs(atan2(dy, dx) - A.reset_psi);
    fwd = c.desired_direction * (sqrt(dx * dx + dy * dy) * cos(psi_diff) / dt);
  } else if (c.task == TASK_AIMING) {
    is_healthy = healthy_turn;
    double tx = A.waypt[0] - xy_before[0], ty = A.waypt[1] - xy_before[1], n = sqrt(tx * tx + ty * ty);
    double target_psi = atan2(ty / n, tx / n);
    double newp = angle_normalize(target_psi - psi_after);
    heading_push(A, newp);
    if (A.head_n > delay) {
      double oldp = heading_pop(A);
      fwd = -(fabs(newp) - fabs(oldp)) / (dt * delay) * c.yaw_reward_weight;
    }
    healthy = 0;
    extra_term = A.step_num > 1000;
  } else if (c.task == TASK_TRACKING) {
    fwd = ditch_reward(c, A, P.xy) - ditch_reward(c, A, xy_before);
    healthy = 0;
    extra_term = A.step_num > 1000;
  } else {  // vel_track, tr_env.py:461-474, 669-678
    double ang = angle_normalize(psi_after - psi_before) / dt;
    double cx = 0.5 * cos(A.reset_psi), cy = 0.5 * sin(A.reset_psi);
    double le = sqrt((xvel - cx) * (xvel - cx) + (yvel - cy) * (yvel - cy)), ae = ang - 0.0;
    fwd = 1.0 * exp(-5.0 * le * le) + 0.5 * exp(-7.0 * ae * ae);
  }
  bool terminated = c.terminate_when_unhealthy ? !is_healthy : false;
  if (extra_term) terminated = true;
  double maxc = 0;
  for (int i = 0; i < 24; i++) maxc = fmax(maxc, fabs((double)S.cfrc[i]));
  if (maxc > c.kill_force) terminated = true;  // tr_env.py:480-481
  double costs = ctrl_cost, info_ctrl = -ctrl_cost;
  if (c.use_contact_forces) {   // tr_env.py:292-304, 513-516
    double cs = 0;
    for (int i = 0; i < 24; i++) { double f = fmin(c.contact_force_range[1], fmax(c.contact_force_range[0], (double)S.cfrc[i])); cs += f * f; }
    cs *= c.contact_cost_weight;
    costs += cs; info_ctrl = -cs;
  }
  O.reward = fwd + healthy - costs;
  O.info_ctrl = info_ctrl;
  O.fwd = fwd; O.ctrl_cost = ctrl_cost; O.healthy = healthy; O.psi = psi_info;
  O.xy[0] = P.xy[0]; O.xy[1] = P.xy[1];
  O.terminated = terminated ? 1 : 0; O.maxcfrc = maxc; O.barforce = (double)S.barforce;
  A.step_num += 1;
  A.xy_prev[0] = P.xy[0]; A.xy_prev[1] = P.xy[1]; A.psi_prev = P.psi;
}

// one env.step(action) with the action in S.action -- warp-collective; obs NOT computed here
template <typename PR>
TB_FN void env_step(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const LaneCtx& L, bool on, Aux& A, StepOut& O, bool aligned) {
  const bool l0 = on && L.bar == 0;
  if (l0) {
    if (c.env_kind == ENV_TR) {  // _action_filter, k_FILTER = 1 (tr_env.py:680-683)
      for (int i = 0; i < NACT; i++) S.ctrl[i] = S.ctrl[i] + 1.0 * (S.action[i] - S.ctrl[i]) * c.dt;
    } else for (int i = 0; i < NACT; i++) S.ctrl[i] = S.action[i];
  }
  wsync();
  simulate(S, m, L, on, c.frame_skip, true, aligned);
  if (l0) env_step_post(S, c, A, O);
  wsync();
}
// refresh the "stale" pose bookkeeping after a forward pass (set_state) -- lane 0
template <typename PR> TB_FN void aux_from_forward(const EnvSh<PR>& S, Aux& A) {
  Pose P; read_pose(S, P);
  A.xy_prev[0] = P.xy[0]; A.xy_prev[1] = P.xy[1]; A.psi_prev = P.psi;
}

// env.reset() = MujocoEnv.reset (mj_resetData) + reset_model, in three pieces so that it can run either in one go
// (tsg_reset) or one warm-up step per launch on a background pool slot.  Random draws: A.draws.
template <typename PR> TB_FN void reset_setpoints(EnvSh<PR>& S, const EnvCfg& c, const Aux& A) {  // lane 0
  const double* u = A.draws;
  for (int i = 0; i < NACT; i++) {
    double t = u[2 + i] * c.tendon_reset_stdev + c.tendon_reset_mean;
    if (t > c.tendon_max_length) t = c.tendon_max_length; else if (t < c.tendon_min_length) t = c.tendon_min_length;
    S.action[i] = t;
  }
}
template <typename PR>
TB_FN void reset_begin(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const LaneCtx& L, bool on, Aux& A) {
  const bool l0 = on && L.bar == 0;
  const double* u = A.draws;
  int idx = 0;
  if (l0) {
    // mj_resetData
    for (int i = 0; i < NV; i++) { S.u.home.qvel[i] = 0; S.u.home.warm[i] = 0; }
    for (int i = 0; i < NACT; i++) { S.ctrl[i] = 0; S.act[i] = 0; }
    idx = (int)floor(u[0] * c.npose);
    if (idx > c.npose - 1) idx = c.npose - 1;
    if (idx < 0) idx = 0;
    for (int i = 0; i < NQ; i++) S.u.home.qpos[i] = c.reset_pose[idx][i];
    if (c.reset_noise_scale > 0) {
      for (int i = 0; i < NQ; i++) S.u.home.qpos[i] += c.reset_noise_scale * reset_noise_draw(A.nz_seed, A.nz_stream, A.nz_nreset, i);
      for (int i = 0; i < NV; i++) S.u.home.qvel[i] = c.reset_noise_scale * reset_noise_draw(A.nz_seed, A.nz_stream, A.nz_nreset, NQ + i);
    }
  }
  wsync();
  bool extra_set_state = (c.env_kind == ENV_TR) ? (c.task == TASK_TURN || c.task == TASK_TRACKING || c.task == TASK_AIMING)
                                                 : (c.task == TASK_TURN);
  int nfwd = (c.env_kind == ENV_TR ? 1 : 0) + (extra_set_state ? 1 : 0);
  for (int k = 0; k < nfwd; k++) simulate(S, m, L, on, 1, false, false);  // set_state -> mj_forward
  if (l0) {
    // rotate the whole robot about world z by theta (positions and orientations), starting again from the table
    // pose: mj_kinematics normalised qpos in place, the reference re-uses its own copy
    double theta = c.min_reset_heading + u[1] * (c.max_reset_heading - c.min_reset_heading);
    double ct = cos(theta), st = sin(theta), ch = cos(0.5 * theta), sh = sin(0.5 * theta);
    for (int b = 0; b < NBAR; b++) {
      double p[7];
      for (int k = 0; k < 7; k++) {
        p[k] = c.reset_pose[idx][7 * b + k];
        if (c.reset_noise_scale > 0) p[k] += c.reset_noise_scale * reset_noise_draw(A.nz_seed, A.nz_stream, A.nz_nreset, 7 * b + k);
      }
      double* q = S.u.home.qpos + 7 * b;
      q[0] = ct * p[0] - st * p[1]; q[1] = st * p[0] + ct * p[1]; q[2] = p[2];
      double n = sqrt(p[3] * p[3] + p[4] * p[4] + p[5] * p[5] + p[6] * p[6]);
      double w = p[3] / n, x = p[4] / n, y = p[5] / n, z = p[6] / n;
      q[3] = ch * w - sh * z; q[4] = ch * x - sh * y; q[5] = ch * y + sh * x; q[6] = ch * z + sh * w;  // q_z(theta) * q
    }
  }
  wsync();
  simulate(S, m, L, on, 1, false, false);
  if (l0) {
    aux_from_forward(S, A);
    reset_setpoints(S, c, A);
    if (c.env_kind == ENV_TR) for (int i = 0; i < NACT; i++) S.ctrl[i] = S.action[i];
  }
  wsync();
}
// one of the warmup_steps settling steps at the set-points in S.action
template <typename PR>
TB_FN void reset_warm_step(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const LaneCtx& L, bool on, Aux& A) {
  if (c.env_kind == ENV_TR) {   // do_simulation, no filter
    simulate(S, m, L, on, c.frame_skip, true, false);
    if (on && L.bar == 0) aux_from_forward(S, A);
    wsync();
  } else { StepOut O; env_step(S, m, c, L, on, A, O, false); }   // full self.step
}
template <typename PR>
TB_FN void reset_finish(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const LaneCtx& L, bool on, Aux& A) {
  if (on && L.bar == 0) {
    const double* u = A.draws;
    Pose P; read_pose(S, P);
    A.reset_psi = P.psi;
    double lo = c.waypt_range[0], hi = c.waypt_range[1];
    if (c.env_kind == ENV_TR && c.task == TASK_TRACKING) {
      A.ori[0] = (P.left[0] + P.right[0]) / 2; A.ori[1] = (P.left[1] + P.right[1]) / 2;
      double len = lo + u[8] * (hi - lo);
      double yaw = c.waypt_angle_range[0] + u[9] * (c.waypt_angle_range[1] - c.waypt_angle_range[0]) + A.reset_psi;
      if (c.is_test) { len = 0.5 * hi + 0.5 * lo; yaw = (0.5 * c.waypt_angle_range[1] + 0.5 * c.waypt_angle_range[0]) + A.reset_psi; }
      A.waypt[0] = A.ori[0] + len * cos(yaw); A.waypt[1] = A.ori[1] + len * sin(yaw);
    } else if (c.env_kind == ENV_TR && c.task == TASK_AIMING) {
      A.ori[0] = P.left[0] + P.right[0] / 2;  // operator-precedence quirk kept (tr_env.py:843)
      A.ori[1] = (P.left[1] + P.right[1]) / 2;
      double len = lo + u[8] * (hi - lo);
      double yaw = -PI + u[9] * (2 * PI) + A.reset_psi;
      if (c.is_test) { len = 0.5 * hi + 0.5 * lo; yaw = (0.75 * PI + 0.25 * (-PI)) + A.reset_psi; }
      A.waypt[0] = A.ori[0] + len * cos(yaw); A.waypt[1] = A.ori[1] + len * sin(yaw);
      if (c.is_test) { A.waypt[0] = 0; A.waypt[1] = 0; }
    }
    A.step_num = 0;
  }
  wsync();
  if (c.env_kind == ENV_TR && (c.task == TASK_TURN || c.task == TASK_AIMING)) {
    StepOut O;
    for (int k = 0; k < c.reward_delay_steps; k++) env_step(S, m, c, L, on, A, O, false);
  }
  if (on && L.bar == 0) { A.ep_ret = 0; A.ep_len = 0; }
}

// ---- state record <-> shared-memory home (the three lanes of the env split the 69 values)
template <typename PR> TB_FN void load_env(EnvSh<PR>& S, const LaneCtx& L, bool on, Aux& A, const double* rec, double* head) {
  if (on) {
    for (int i = L.bar; i < SO_XY_PREV; i += G) {
      double v = rec[i];
      if (i < SO_QVEL) S.u.home.qpos[i] = v;
      else if (i < SO_WARM) S.u.home.qvel[i - SO_QVEL] = v;
      else if (i < SO_CTRL) S.u.home.warm[i - SO_WARM] = v;
      else if (i < SO_ACT) S.ctrl[i - SO_CTRL] = v;
      else S.act[i - SO_ACT] = v;
    }
    if (L.bar == 0) {
      A.heading = head;
      A.xy_prev[0] = rec[SO_XY_PREV]; A.xy_prev[1] = rec[SO_XY_PREV + 1]; A.psi_prev = rec[SO_PSI_PREV];
      A.reset_psi = rec[SO_RESET_PSI]; A.waypt[0] = rec[SO_WAYPT]; A.waypt[1] = rec[SO_WAYPT + 1];
      A.ori[0] = rec[SO_ORI]; A.ori[1] = rec[SO_ORI + 1];
      A.step_num = rec[SO_STEP_NUM]; A.ep_ret = rec[SO_EP_RET]; A.ep_len = rec[SO_EP_LEN];
      A.xvel = rec[SO_XVEL]; A.yvel = rec[SO_YVEL];
      A.head_n = (int)rec[SO_HEAD_N]; A.head_pos = (int)rec[SO_HEAD_POS];
      S.overflow = 0; S.bad = 0; S.niter = 0; S.nls = 0; S.nmpr = 0; S.nact = 0; S.barforce = 0;
    }
  }
  wsync();
}
template <typename PR> TB_FN void store_env(const EnvSh<PR>& S, const LaneCtx& L, bool on, const Aux& A, double* rec) {
  if (!on) return;
  for (int i = L.bar; i < SO_XY_PREV; i += G) {
    double v;
    if (i < SO_QVEL) v = S.u.home.qpos[i];
    else if (i < SO_WARM) v = S.u.home.qvel[i - SO_QVEL];
    else if (i < SO_CTRL) v = S.u.home.warm[i - SO_WARM];
    else if (i < SO_ACT) v = S.ctrl[i - SO_CTRL];
    else v = S.act[i - SO_ACT];
    rec[i] = v;
  }
  if (L.bar == 0) {
    rec[SO_XY_PREV] = A.xy_prev[0]; rec[SO_XY_PREV + 1] = A.xy_prev[1]; rec[SO_PSI_PREV] = A.psi_prev;
    rec[SO_RESET_PSI] = A.reset_psi; rec[SO_WAYPT] = A.waypt[0]; rec[SO_WAYPT + 1] = A.waypt[1];
    rec[SO_ORI] = A.ori[0]; rec[SO_ORI + 1] = A.ori[1];
    rec[SO_STEP_NUM] = A.step_num; rec[SO_EP_RET] = A.ep_ret; rec[SO_EP_LEN] = A.ep_len;
    rec[SO_XVEL] = A.xvel; rec[SO_YVEL] = A.yvel;
    rec[SO_HEAD_N] = (double)A.head_n; rec[SO_HEAD_POS] = (double)A.head_pos;
  }
}

TB_FN void write_obs(const EnvCfg& c, const StepIO& io, int e, const double* obs) {   // lane 0
  if (io.obs) for (int i = 0; i < c.obs_dim; i++) io.obs[(size_t)e * c.obs_dim + i] = obs[i];
  if (io.obs32) for (int i = 0; i < c.obs_dim; i++) io.obs32[(size_t)e * c.obs_dim + i] = (float)obs[i];
}
TB_FN void make_draws(double* d, unsigned long long seed, unsigned long long env_id, unsigned long long nreset) {
  double un[12];
  for (int k = 0; k < 6; k++) {
    uint32_t r[4];
    philox(seed, env_id, (nreset << 8) | (unsigned long long)k, r);
    un[2 * k] = u01(r[0], r[1]); un[2 * k + 1] = u01(r[2], r[3]);
  }
  d[0] = un[0]; d[1] = un[1]; d[8] = un[2]; d[9] = un[3];
  for (int k = 0; k < 3; k++) {  // Box-Muller
    double u1 = 1.0 - un[4 + 2 * k], u2 = un[5 + 2 * k];
    double r = sqrt(-2.0 * log(u1));
    d[2 + 2 * k] = r * cos(2 * PI * u2); d[3 + 2 * k] = r * sin(2 * PI * u2);
  }
}

// Per-env parameter row of a reset: row[i] = nominal[i] * U(lo[i], hi[i]), prange = {nominal, lo, hi}[NPARAM].  Draw j
// of the 32 is u01 half j & 1 of Philox(seed ^ key, stream, (nreset << 8) | j / 2); the lower and upper spring length
// of a tendon share one draw, so a deadband stays ordered.  The scale is rounded before the product (no fused
// multiply-add) so that the host emulator draws the same rows bit for bit.
TB_FN double draw_param(const double* prange, unsigned long long seed, unsigned long long stream, unsigned long long nreset, int i) {
  const int j = i < PRM_TLS ? i : (i < PRM_GAIN ? PRM_TLS + (i - PRM_TLS) / 2 : i - NTEN);
  uint32_t r[4];
  philox(seed ^ 0x706172616d726e64ull, stream, (nreset << 8) | (unsigned long long)(j >> 1), r);
  const double u = (j & 1) ? u01(r[2], r[3]) : u01(r[0], r[1]);
  const double lo = prange[NPARAM + i], hi = prange[2 * NPARAM + i];
#if TB_DEV
  const double scale = __dadd_rn(lo, __dmul_rn(u, hi - lo));
#else
  const double scale = lo + u * (hi - lo);
#endif
  return prange[i] * scale;
}
TB_FN void draw_params(double* row, const double* prange, unsigned long long seed, unsigned long long stream, unsigned long long nreset) {
  for (int i = 0; i < NPARAM; i++) row[i] = draw_param(prange, seed, stream, nreset, i);
}
// per-env variant: point the env's slice at its parameter row (lane 0; the caller's next wsync publishes it)
template <typename PR> TB_FN void set_prm_row(EnvSh<PR>& S, const StepIO& io, size_t row) {
  if constexpr (PR::per_env) S.prm = io.params + row * NPARAM;
}

constexpr int OBS_MAX = 160;

// ---- the step of EPW consecutive envs starting at `first` (one warp)
template <typename PR>
TB_FN void run_step(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const StepIO& io, const LaneCtx& L, int first, bool aligned) {
  const int e = first + L.grp;
  const bool on = L.valid && e < io.n_envs, l0 = on && L.bar == 0;
  Aux A; StepOut O;
  double* rec = io.state + (size_t)(on ? e : 0) * STATE_STRIDE;
  load_env(S, L, on, A, rec, io.heading + (size_t)(on ? e : 0) * HEADING_SLOTS);
  if (l0) {
    for (int i = 0; i < NACT; i++) S.action[i] = io.ctrl64 ? io.ctrl64[(size_t)e * NACT + i] : (double)io.ctrl32[(size_t)e * NACT + i];
    set_prm_row(S, io, (size_t)e);
  }
  wsync();
  env_step(S, m, c, L, on, A, O, aligned);
  if (l0) {
    double obs[OBS_MAX];
    compute_obs(S, c, A, obs);
    A.ep_len += 1; A.ep_ret += O.reward;
    if (c.use_obs_noise) {
      if (io.real_obs) for (int i = 0; i < c.obs_dim; i++) io.real_obs[(size_t)e * c.obs_dim + i] = obs[i];
      obs_noise(c, obs, io.seed, (unsigned long long)(io.env_id_base + e), (unsigned long long)rec[SO_NRESET], (unsigned long long)A.ep_len);
    }
    int truncated = (c.max_episode_steps > 0 && A.ep_len >= c.max_episode_steps) ? 1 : 0;
    write_obs(c, io, e, obs);
    if (io.reward) io.reward[e] = O.reward;
    if (io.done) io.done[e] = (uint8_t)((O.terminated || truncated) ? 1 : 0);
    if (io.info) {
      double* I = io.info + (size_t)e * INFO_DIM;
      for (int i = 0; i < INFO_DIM; i++) I[i] = 0;
      I[IO_REW_FWD] = O.fwd; I[IO_REW_CTRL] = O.info_ctrl; I[IO_REW_SURVIVE] = O.healthy;
      I[IO_X] = O.xy[0]; I[IO_Y] = O.xy[1]; I[IO_PSI] = O.psi; I[IO_XVEL] = A.xvel; I[IO_YVEL] = A.yvel;
      for (int i = 0; i < 9; i++) I[IO_TEN + i] = (double)S.tlen[i];
      I[IO_TERMINATED] = O.terminated; I[IO_TRUNCATED] = truncated;
      I[IO_NCON] = S.nact; I[IO_NITER] = S.niter; I[IO_NLS] = S.nls; I[IO_BARFORCE] = O.barforce; I[IO_MAXCFRC] = O.maxcfrc;
      I[IO_WAYPT] = A.waypt[0]; I[IO_WAYPT + 1] = A.waypt[1]; I[IO_ORI] = A.ori[0]; I[IO_ORI + 1] = A.ori[1];
      I[IO_OVERFLOW] = S.overflow; I[IO_BAD] = S.bad; I[IO_NMPR] = S.nmpr; I[IO_RESET_PSI] = A.reset_psi;
    }
  }
  wsync();
  store_env(S, L, on, A, rec);
  wsync();
}

// ---- reset of the masked envs among EPW consecutive ones
template <typename PR>
TB_FN void run_reset(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const StepIO& io, const LaneCtx& L, int first) {
  const int e = first + L.grp;
  const bool on = L.valid && e < io.n_envs && (!io.mask || io.mask[e]), l0 = on && L.bar == 0;
  if (!any(on)) return;
  Aux A;
  double* rec = io.state + (size_t)(on ? e : 0) * STATE_STRIDE;
  load_env(S, L, on, A, rec, io.heading + (size_t)(on ? e : 0) * HEADING_SLOTS);
  double nreset = 0;
  if (l0) {
    if (io.term_obs && io.obs) for (int i = 0; i < c.obs_dim; i++) io.term_obs[(size_t)e * c.obs_dim + i] = io.obs[(size_t)e * c.obs_dim + i];
    nreset = rec[SO_NRESET];
    double* dr = io.draws + (size_t)e * NDRAW;
    if (!io.explicit_draws) make_draws(dr, io.seed, (unsigned long long)(io.env_id_base + e), (unsigned long long)nreset);
    A.draws = dr;
    A.nz_seed = io.seed; A.nz_stream = (unsigned long long)(io.env_id_base + e); A.nz_nreset = (unsigned long long)nreset;
    if constexpr (PR::per_env) {
      set_prm_row(S, io, (size_t)e);
      if (io.prange) draw_params(io.params + (size_t)e * NPARAM, io.prange, io.seed, A.nz_stream, A.nz_nreset);
    }
  }
  wsync();
  reset_begin(S, m, c, L, on, A);
  for (int k = 0; k < c.warmup_steps; k++) reset_warm_step(S, m, c, L, on, A);
  reset_finish(S, m, c, L, on, A);
  if (l0) {
    double obs[OBS_MAX];
    compute_obs(S, c, A, obs);
    if (c.use_obs_noise) {
      if (io.real_obs) for (int i = 0; i < c.obs_dim; i++) io.real_obs[(size_t)e * c.obs_dim + i] = obs[i];
      obs_noise(c, obs, io.seed, (unsigned long long)(io.env_id_base + e), (unsigned long long)(nreset + 1), 0ull);
    }
    write_obs(c, io, e, obs);
  }
  wsync();
  store_env(S, L, on, A, rec);
  if (l0) rec[SO_NRESET] = nreset + 1;
  wsync();
}

// ---- background reset pool: slot p (record n_envs + p) advances by one warm-up step per launch until it holds a
// completely reset env (state, heading ring, reset observation); tsg_assign_kernel then hands ready slots to envs
// that are done.  phase (SO_FLAGS) = warm-up steps done, warmup_steps + 1 = ready.  finish_now: run to completion.
template <typename PR>
TB_FN void run_pool(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const StepIO& io, const LaneCtx& L, int first, bool finish_now) {
  const int p = first + L.grp;
  const bool valid = L.valid && p < io.n_pool;
  const size_t row = (size_t)io.n_envs + (valid ? p : 0);
  double* rec = io.state + row * STATE_STRIDE;
  int phase = valid ? (int)rec[SO_FLAGS] : c.warmup_steps + 1;
  const bool on = valid && phase <= c.warmup_steps, l0 = on && L.bar == 0;
  if (!any(on)) return;
  Aux A;
  load_env(S, L, on, A, rec, io.heading + row * HEADING_SLOTS);
  double nreset = 0;
  if (l0) {
    nreset = rec[SO_NRESET];
    double* dr = io.draws + row * NDRAW;
    if (phase == 0) make_draws(dr, io.seed, (1ull << 40) + (unsigned long long)(io.env_id_base + p), (unsigned long long)nreset);
    A.draws = dr;
    A.nz_seed = io.seed; A.nz_stream = (1ull << 40) + (unsigned long long)(io.env_id_base + p); A.nz_nreset = (unsigned long long)nreset;
    if constexpr (PR::per_env) {   // the slot's row; tsg_assign hands it to the env together with the record
      set_prm_row(S, io, row);
      if (phase == 0 && io.prange) draw_params(io.params + row * NPARAM, io.prange, io.seed, A.nz_stream, A.nz_nreset);
    }
  }
  wsync();
  const bool begin = on && phase == 0;
  if (any(begin)) reset_begin(S, m, c, L, begin, A);
  if (l0 && phase != 0) reset_setpoints(S, c, A);
  wsync();
  bool warming = on;
  do {
    reset_warm_step(S, m, c, L, warming, A);
    if (warming) phase++;
    warming = warming && finish_now && phase < c.warmup_steps;
  } while (any(warming));
  const bool fin = on && phase >= c.warmup_steps;
  if (any(fin)) {
    reset_finish(S, m, c, L, fin, A);
    if (fin && L.bar == 0) {
      double obs[OBS_MAX];
      compute_obs(S, c, A, obs);
      if (c.use_obs_noise) {
        if (io.pool_real_obs) for (int i = 0; i < c.obs_dim; i++) io.pool_real_obs[(size_t)p * c.obs_dim + i] = obs[i];
        obs_noise(c, obs, io.seed, (1ull << 40) + (unsigned long long)(io.env_id_base + p), (unsigned long long)(nreset + 1), 0ull);
      }
      for (int i = 0; i < c.obs_dim; i++) io.pool_obs[(size_t)p * c.obs_dim + i] = obs[i];
    }
    if (fin) phase = c.warmup_steps + 1;
  }
  wsync();
  store_env(S, L, on, A, rec);
  if (l0) rec[SO_FLAGS] = (double)phase;
  wsync();
}

// ---- mj_forward on the stored state (after tsg_set_state): refresh kinematics bookkeeping and obs
template <typename PR>
TB_FN void run_forward(EnvSh<PR>& S, const ModelT<typename PR::real>& m, const EnvCfg& c, const StepIO& io, const LaneCtx& L, int first) {
  const int e = first + L.grp;
  const bool on = L.valid && e < io.n_envs, l0 = on && L.bar == 0;
  Aux A;
  double* rec = io.state + (size_t)(on ? e : 0) * STATE_STRIDE;
  load_env(S, L, on, A, rec, io.heading + (size_t)(on ? e : 0) * HEADING_SLOTS);
  if constexpr (PR::per_env) {
    if (l0) set_prm_row(S, io, (size_t)e);
    wsync();
  }
  simulate(S, m, L, on, 1, false, false);
  if (l0) {
    aux_from_forward(S, A);
    double obs[OBS_MAX];
    compute_obs(S, c, A, obs);
    write_obs(c, io, e, obs);
    if (io.info) {
      double* I = io.info + (size_t)e * INFO_DIM;
      for (int i = 0; i < INFO_DIM; i++) I[i] = 0;
      for (int i = 0; i < 9; i++) I[IO_TEN + i] = (double)S.tlen[i];
      I[IO_NCON] = S.nact; I[IO_X] = A.xy_prev[0]; I[IO_Y] = A.xy_prev[1]; I[IO_PSI] = A.psi_prev;
      I[IO_BARFORCE] = (double)S.barforce;
    }
  }
  wsync();
  store_env(S, L, on, A, rec);
  wsync();
}

}  // namespace tb
