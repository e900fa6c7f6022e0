// tb_model.h -- device-side constants of the bar-lane kernel and their host-side preparation from the C-ABI structs
// (include/tsg_model.h).  ModelT<real> is what MjModel.from_xml_path() yields for the two reference XMLs, cut down to
// the fields the hot path reads and pre-digested (inverse masses, impedance constants, per-bar tendon-end lists).
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <string>

#include "../../include/tsg_model.h"

namespace tb {

constexpr int NBAR = 3, NGEOM = 15, NTEN = 9, NEND = 18, NACT = 6, NQ = 21, NV = 18;
constexpr int GEOM_SPHERE = 2, GEOM_CYL = 5;
constexpr int STATE_STRIDE = 96;  // doubles per env record in HBM (768 B, 128 B aligned)
constexpr int INFO_DIM = 32;
constexpr int HEADING_SLOTS = 32;
constexpr int NDRAW = 10;
constexpr double PI = 3.14159265358979323846;
// per-env parameter row (include/tsg.h TSG_PARAM_*): absolute values in model units
constexpr int NPARAM = 41;
enum ParamOff { PRM_TK = 0, PRM_TDAMP = 9, PRM_TLS = 18 /* lower, upper per tendon */, PRM_GAIN = 36, PRM_BIAS = 37, PRM_DYNPRM0 = 40 };
enum { ENV_TR = 0, ENV_LEGACY = 1 };
enum { TASK_STRAIGHT = 0, TASK_TURN = 1, TASK_AIMING = 2, TASK_TRACKING = 3, TASK_VEL_TRACK = 4 };

// offsets into the per-env state record
enum StateOff {
  SO_QPOS = 0, SO_QVEL = 21, SO_WARM = 39, SO_CTRL = 57, SO_ACT = 63,
  SO_XY_PREV = 69, SO_PSI_PREV = 71, SO_RESET_PSI = 72, SO_WAYPT = 73, SO_ORI = 75,
  SO_STEP_NUM = 77, SO_EP_RET = 78, SO_EP_LEN = 79, SO_XVEL = 80, SO_YVEL = 81,
  SO_HEAD_N = 82, SO_HEAD_POS = 83, SO_FLAGS = 84, SO_NRESET = 85, SO_USED = 86
};
// info row (per env, per step)
enum InfoOff {
  IO_REW_FWD = 0, IO_REW_CTRL, IO_REW_SURVIVE, IO_X, IO_Y, IO_PSI, IO_XVEL, IO_YVEL,
  IO_TEN = 8 /* 9 */, IO_TERMINATED = 17, IO_TRUNCATED, IO_NCON, IO_NITER, IO_NLS, IO_BARFORCE, IO_MAXCFRC,
  IO_WAYPT = 24 /* 2 */, IO_ORI = 26 /* 2 */, IO_OVERFLOW = 28, IO_BAD = 29, IO_NMPR = 30, IO_RESET_PSI = 31
};

template <typename real>
struct ModelT {
  real h, grav[3], tol, ls_tol, mpr_tol, meaninertia;
  real solscale;   // 1 / (meaninertia * nv): scale of the solver's convergence tests
  real gradtol;    // tol * meaninertia * nv
  int iterations, ls_iterations, mpr_iterations;
  unsigned flags;
  real M[NV], invM[NV];
  real inertia[NBAR][3];
  real invw_tran[NBAR];
  int gtype[NGEOM];
  int pad0;
  real gsize[NGEOM][2];
  real gpos[NGEOM][3];
  real gbound[NGEOM];   // bounding-sphere radius of the geom about its centre
  real gz[NGEOM];       // position of the geom's centre along the bar axis (all geoms lie on it)
  // tendons
  int tbody[NEND];
  real tsite[NEND][3];
  real tk[NTEN], tdamp[NTEN], tls[NTEN][2];
  int ten_act[NTEN];
  int nends[NBAR];
  int ends[NBAR][8];
  int dyntype, ctrllimited, forcelimited, pad1;
  real dynprm0, gain, bias[3], ctrlrange[2], forcerange[2];
  // contact
  real K, B, solimp[5], mu, fr[5], dscale[6];
  real wtab[2][6];   // Hessian row weights per zone: bottom = dscale, middle = (0, fr^2)
  real inv_mu2;      // 1 / (mu^2 (1 + mu^2))
  // floor
  int floor_type, nrow, ncol, pad2;
  real fpos[3], fnormal[3], hsize[4];
  real hdx, hdy;     // height-field cell size
  const float* hdata;
  real qpos0[NQ];
};

struct EnvCfg {
  int env_kind, task, frame_skip, obs_dim, use_cap_velocity, terminate_when_unhealthy, is_test;
  int reward_delay_steps, max_episode_steps, warmup_steps, npose, use_obs_noise, use_contact_forces, pad_;
  double desired_direction, ctrl_cost_weight, healthy_reward, yaw_reward_weight;
  double min_reset_heading, max_reset_heading;
  double tendon_reset_mean, tendon_reset_stdev, tendon_min_length, tendon_max_length;
  double waypt_range[2], waypt_angle_range[2];
  double ditch_reward_max, ditch_reward_stdev, waypt_reward_amplitude, waypt_reward_stdev, kill_force, dt;
  double obs_noise_tendon_stdev, obs_noise_cap_pos_stdev;
  double reset_noise_scale, contact_cost_weight, contact_force_range[2];
  double reset_pose[6][NQ];
};

constexpr double MINVAL_D = 1e-15, MAXVAL_D = 1e10, MINIMP_D = 0.0001, MAXIMP_D = 0.9999;

// returns "" on success, else an error message
template <typename real>
inline std::string make_model(const TsgModel& t, ModelT<real>& m, const float* hdata_dev) {
  if (t.struct_bytes != (int)sizeof(TsgModel)) return "TsgModel.struct_bytes mismatch";
  memset(&m, 0, sizeof(m));
  m.h = (real)t.timestep;
  for (int k = 0; k < 3; k++) m.grav[k] = (real)t.gravity[k];
  m.tol = (real)t.tolerance; m.ls_tol = (real)t.ls_tolerance; m.mpr_tol = (real)t.mpr_tolerance; m.meaninertia = (real)t.meaninertia;
  m.iterations = t.iterations; m.ls_iterations = t.ls_iterations; m.mpr_iterations = t.mpr_iterations;
  m.flags = t.flags;
  if (t.flags & TSG_FLAG_CROSSBAR_DERIV) return "TSG_FLAG_CROSSBAR_DERIV is an oracle-only switch";
  for (int b = 0; b < NBAR; b++) {
    for (int j = 0; j < 6; j++) {
      double M = j < 3 ? t.body_mass[b] : t.body_inertia[b][j - 3];
      m.M[6 * b + j] = (real)M; m.invM[6 * b + j] = (real)(1.0 / M);
    }
    for (int k = 0; k < 3; k++) m.inertia[b][k] = (real)t.body_inertia[b][k];
    m.invw_tran[b] = (real)t.body_invweight0[b][0];
    for (int g = 0; g < 5; g++) {
      int G = 5 * b + g;
      m.gtype[G] = t.geom_type[b][g];
      if (m.gtype[G] != GEOM_SPHERE && m.gtype[G] != GEOM_CYL) return "geom type must be sphere or cylinder";
      double r = t.geom_size[b][g][0], hl = t.geom_size[b][g][1];
      m.gsize[G][0] = (real)r; m.gsize[G][1] = (real)hl;
      m.gbound[G] = (real)(m.gtype[G] == GEOM_SPHERE ? r : sqrt(r * r + hl * hl));
      for (int k = 0; k < 3; k++) m.gpos[G][k] = (real)t.geom_pos[b][g][k];
      if (t.geom_pos[b][g][0] != 0 || t.geom_pos[b][g][1] != 0) return "geoms must be centred on the bar axis";
      m.gz[G] = (real)t.geom_pos[b][g][2];
      // geom frames must be the body frame up to axis flips (cylinders/spheres are symmetric under those)
      const double* q = t.geom_quat[b][g];
      int big = 0;
      for (int k = 0; k < 4; k++) if (fabs(q[k]) > 1 - 1e-9) big++;
      if (big != 1) return "geom quaternions must be axis flips of the body frame";
    }
  }
  for (int k = 0; k < NQ; k++) m.qpos0[k] = (real)t.qpos0[k];
  for (int b = 0; b < NBAR; b++) m.nends[b] = 0;
  for (int tt = 0; tt < NTEN; tt++) {
    m.ten_act[tt] = -1;
    m.tk[tt] = (real)t.ten_stiffness[tt]; m.tdamp[tt] = (real)t.ten_damping[tt];
    m.tls[tt][0] = (real)t.ten_lengthspring[tt][0]; m.tls[tt][1] = (real)t.ten_lengthspring[tt][1];
    if (t.ten_body[tt][0] == t.ten_body[tt][1]) return "tendon sites must be on different bars";
    for (int e = 0; e < 2; e++) {
      int end = 2 * tt + e, b = t.ten_body[tt][e];
      if (b < 0 || b >= NBAR) return "bad tendon body";
      m.tbody[end] = b;
      for (int k = 0; k < 3; k++) m.tsite[end][k] = (real)t.ten_site[tt][e][k];
      if (m.nends[b] >= 8) return "too many tendon ends on one bar";
      m.ends[b][m.nends[b]++] = end;
    }
  }
  for (int a = 0; a < NACT; a++) {
    if (t.act_tendon[a] < 0 || t.act_tendon[a] >= NTEN || m.ten_act[t.act_tendon[a]] >= 0) return "bad actuator tendon";
    m.ten_act[t.act_tendon[a]] = a;
  }
  m.dyntype = t.act_dyntype; m.ctrllimited = t.ctrllimited; m.forcelimited = t.forcelimited;
  m.dynprm0 = (real)t.act_dynprm0; m.gain = (real)t.act_gain;
  for (int k = 0; k < 3; k++) m.bias[k] = (real)t.act_bias[k];
  for (int k = 0; k < 2; k++) { m.ctrlrange[k] = (real)t.ctrlrange[k]; m.forcerange[k] = (real)t.forcerange[k]; }
  if (!(t.solref[0] < 0 && t.solref[1] < 0)) return "only direct (negative) solref is supported";
  if (t.condim != 6) return "condim must be 6";
  if (t.friction[0] != t.friction[1] || t.friction[3] != t.friction[4]) return "friction must be isotropic (slide, slide, spin, roll, roll)";
  double dmax = fmin(MAXIMP_D, fmax(MINIMP_D, t.solimp[1]));
  m.K = (real)(-t.solref[0] / (dmax * dmax)); m.B = (real)(-t.solref[1] / dmax);
  for (int k = 0; k < 5; k++) { m.solimp[k] = (real)t.solimp[k]; m.fr[k] = (real)t.friction[k]; }
  double mu = t.friction[0] / sqrt(t.impratio);
  m.mu = (real)mu;
  m.inv_mu2 = (real)(1.0 / (mu * mu * (1 + mu * mu)));
  m.solscale = (real)(1.0 / (t.meaninertia * NV));
  m.gradtol = (real)(t.tolerance * t.meaninertia * NV);
  m.dscale[0] = 1;
  for (int j = 1; j < 6; j++)   // R_j = (R_0 / impratio) * f0^2 / f_{j-1}^2  ->  D_j = D_0 * dscale_j
    m.dscale[j] = (real)(t.impratio * (t.friction[j - 1] * t.friction[j - 1]) / (t.friction[0] * t.friction[0]));
  for (int r = 0; r < 6; r++) { m.wtab[0][r] = m.dscale[r]; m.wtab[1][r] = (real)(r ? t.friction[r - 1] * t.friction[r - 1] : 0.0); }
  m.floor_type = t.floor_type;
  for (int k = 0; k < 3; k++) { m.fpos[k] = (real)t.floor_pos[k]; m.fnormal[k] = (real)t.floor_mat[3 * k + 2]; }
  if (t.floor_type == TSG_FLOOR_HFIELD) {
    const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int k = 0; k < 9; k++) if (fabs(t.floor_mat[k] - I[k]) > 1e-12) return "height field frame must be axis aligned";
    m.nrow = t.hf_nrow; m.ncol = t.hf_ncol;
    for (int k = 0; k < 4; k++) m.hsize[k] = (real)t.hf_size[k];
    m.hdx = (real)(2.0 * t.hf_size[0] / (double)(m.ncol - 1)); m.hdy = (real)(2.0 * t.hf_size[1] / (double)(m.nrow - 1));
    m.hdata = hdata_dev;
    if (!hdata_dev || m.nrow < 2 || m.ncol < 2) return "height field data missing";
  }
  return "";
}

// the nominal parameter row: the TsgModel fields make_model reads into tk / tdamp / tls / gain / bias / dynprm0
inline void nominal_params(const TsgModel& t, double* row) {
  for (int tt = 0; tt < NTEN; tt++) {
    row[PRM_TK + tt] = t.ten_stiffness[tt]; row[PRM_TDAMP + tt] = t.ten_damping[tt];
    row[PRM_TLS + 2 * tt] = t.ten_lengthspring[tt][0]; row[PRM_TLS + 2 * tt + 1] = t.ten_lengthspring[tt][1];
  }
  row[PRM_GAIN] = t.act_gain;
  for (int k = 0; k < 3; k++) row[PRM_BIAS + k] = t.act_bias[k];
  row[PRM_DYNPRM0] = t.act_dynprm0;
}
// scale ranges of the reset draws, lo / hi [NPARAM]; returns "" when valid
inline std::string check_param_ranges(const double* lo, const double* hi) {
  for (int i = 0; i < NPARAM; i++) {
    if (!isfinite(lo[i]) || !isfinite(hi[i])) return "param ranges must be finite";
    if (!(lo[i] >= 0 && lo[i] <= hi[i])) return "param ranges need 0 <= lo <= hi";
  }
  if (!(lo[PRM_DYNPRM0] > 0)) return "the act_dynprm0 scale must be above 0";
  for (int tt = 0; tt < NTEN; tt++)
    if (lo[PRM_TLS + 2 * tt] != lo[PRM_TLS + 2 * tt + 1] || hi[PRM_TLS + 2 * tt] != hi[PRM_TLS + 2 * tt + 1])
      return "the lower and upper ten_lengthspring of a tendon share one draw: their ranges must be equal";
  return "";
}

inline std::string make_env_cfg(const TsgEnvConfig& t, const TsgModel& mod, EnvCfg& c) {
  if (t.struct_bytes != (int)sizeof(TsgEnvConfig)) return "TsgEnvConfig.struct_bytes mismatch";
  memset(&c, 0, sizeof(c));
  c.env_kind = t.env_kind; c.task = t.task; c.frame_skip = t.frame_skip; c.obs_dim = t.obs_dim;
  c.use_cap_velocity = t.use_cap_velocity; c.terminate_when_unhealthy = t.terminate_when_unhealthy;
  c.is_test = t.is_test; c.reward_delay_steps = t.reward_delay_steps; c.max_episode_steps = t.max_episode_steps;
  c.warmup_steps = t.warmup_steps; c.npose = t.npose;
  if (c.frame_skip < 1) return "frame_skip must be >= 1";
  if (c.obs_dim < 1 || c.obs_dim > 160) return "obs_dim out of range";
  if (c.npose < 1 || c.npose > TSG_NPOSE) return "npose out of range";
  if (c.warmup_steps < 1) return "warmup_steps must be >= 1";
  bool ring = c.task == TASK_TURN || c.task == TASK_AIMING;   // only these tasks use the heading ring
  if (ring && (c.reward_delay_steps < 1 || c.reward_delay_steps + 1 > HEADING_SLOTS)) return "reward_delay_steps out of range";
  if (!ring && c.reward_delay_steps < 1) c.reward_delay_steps = 1;
  if (c.env_kind == ENV_LEGACY && c.task > TASK_TURN) return "tensegrity_env supports straight/turn only";
  c.desired_direction = t.desired_direction; c.ctrl_cost_weight = t.ctrl_cost_weight;
  c.healthy_reward = t.healthy_reward; c.yaw_reward_weight = t.yaw_reward_weight;
  c.min_reset_heading = t.min_reset_heading; c.max_reset_heading = t.max_reset_heading;
  c.tendon_reset_mean = t.tendon_reset_mean; c.tendon_reset_stdev = t.tendon_reset_stdev;
  c.tendon_min_length = t.tendon_min_length; c.tendon_max_length = t.tendon_max_length;
  for (int k = 0; k < 2; k++) { c.waypt_range[k] = t.waypt_range[k]; c.waypt_angle_range[k] = t.waypt_angle_range[k]; }
  c.ditch_reward_max = t.ditch_reward_max; c.ditch_reward_stdev = t.ditch_reward_stdev;
  c.waypt_reward_amplitude = t.waypt_reward_amplitude; c.waypt_reward_stdev = t.waypt_reward_stdev;
  c.kill_force = t.kill_force;
  c.use_obs_noise = t.use_obs_noise ? 1 : 0;
  c.obs_noise_tendon_stdev = t.obs_noise_tendon_stdev; c.obs_noise_cap_pos_stdev = t.obs_noise_cap_pos_stdev;
  if (c.use_obs_noise && c.env_kind != ENV_TR) return "use_obs_noise exists for tr_env only";
  if (c.use_obs_noise && (c.obs_noise_tendon_stdev < 0 || c.obs_noise_cap_pos_stdev < 0)) return "negative obs noise stdev";
  c.reset_noise_scale = t.reset_noise_scale;
  if (!(c.reset_noise_scale >= 0)) return "negative reset_noise_scale";
  c.use_contact_forces = t.use_contact_forces ? 1 : 0;
  c.contact_cost_weight = t.contact_cost_weight;
  c.contact_force_range[0] = t.contact_force_range[0]; c.contact_force_range[1] = t.contact_force_range[1];
  c.dt = mod.timestep * t.frame_skip;
  for (int p = 0; p < TSG_NPOSE; p++) for (int k = 0; k < NQ; k++) c.reset_pose[p][k] = t.reset_pose[p][k];
  return "";
}

}  // namespace tb
