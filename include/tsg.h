/* tsg.h -- C ABI of libtsg.so, the B200-native batched 3-bar tensegrity simulator.
 *
 * This is the drop-in boundary for the reference's hot path.  Each entry point
 * replaces the MuJoCo / gym call the reference's envs make in-process:
 *
 *   tsg_create      <- MjModel.from_xml_path + MjData   (gym MujocoEnv.__init__, tr_env.py:274-276,
 *                                                         tensegrity_env.py:239-241), for N envs
 *   tsg_reset       <- MujocoEnv.reset -> mj_resetData + reset_model (tr_env.py:709-872,
 *                                                         tensegrity_env.py:433-512)
 *   tsg_step        <- env.step: _action_filter + do_simulation (mj_step x frame_skip +
 *                      mj_rnePostConstraint) + _get_obs + reward + termination
 *                      (tr_env.py:327-527, tensegrity_env.py:291-410)
 *   tsg_set_state   <- MujocoEnv.set_state (qpos/qvel write; tr_env.py:744,763,800) and direct
 *                      writes of data.ctrl / data.act / data.qacc_warmstart
 *   tsg_forward     <- mujoco.mj_forward (inside set_state)
 *   tsg_get_state   <- reads of data.qpos / qvel / act / ctrl / qacc_warmstart
 *   info rows       <- the info dict of step (tr_env.py:496-512) + mj_contactForce sum of run.py:155-161
 *
 * Conventions: all functions return 0 on success, <0 on error (tsg_last_error() has the text);
 * no C++ exceptions cross the boundary.  The handle owns the persistent per-env state in HBM;
 * the caller owns every buffer it passes.  Pointers named *_dev are DEVICE pointers valid on the
 * handle's device; `stream` is a cudaStream_t (0 = default) and no call synchronises the host
 * unless it copies to host memory (the *_host variants).  One handle per device / per rank.
 */
#ifndef TSG_H_
#define TSG_H_

#include <stddef.h>
#include <stdint.h>

#include "tsg_model.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct TsgHandle TsgHandle;

#define TSG_STATE_STRIDE 96 /* doubles per env record (qpos 21, qvel 18, warmstart 18, ctrl 6, act 6, aux) */
#define TSG_INFO_DIM 32
#define TSG_CTRL_F64 0
#define TSG_CTRL_F32 1
#define TSG_PRECISION_F64 0 /* the reference's arithmetic (MuJoCo is float64); the default */
#define TSG_PRECISION_F32 1 /* optional fp32 physics (state records, rewards and observations stay f64) */

/* per-env parameter row (doubles, absolute values in model units); the nominal row holds the TsgModel fields of the
 * same names */
#define TSG_NPARAM 41
#define TSG_PARAM_TEN_STIFFNESS 0    /* 9 */
#define TSG_PARAM_TEN_DAMPING 9      /* 9 */
#define TSG_PARAM_TEN_LENGTHSPRING 18 /* 18: lower, upper of tendon 0, then tendon 1, ... */
#define TSG_PARAM_ACT_GAIN 36        /* 1 */
#define TSG_PARAM_ACT_BIAS 37        /* 3 */
#define TSG_PARAM_ACT_DYNPRM0 40     /* 1 */

/* info row layout (doubles) */
#define TSG_INFO_REW_FWD 0
#define TSG_INFO_REW_CTRL 1
#define TSG_INFO_REW_SURVIVE 2
#define TSG_INFO_X 3
#define TSG_INFO_Y 4
#define TSG_INFO_PSI 5
#define TSG_INFO_XVEL 6
#define TSG_INFO_YVEL 7
#define TSG_INFO_TEN 8 /* 9 tendon lengths */
#define TSG_INFO_TERMINATED 17
#define TSG_INFO_TRUNCATED 18
#define TSG_INFO_NCON 19
#define TSG_INFO_NITER 20 /* Newton iterations summed over the substeps of the step */
#define TSG_INFO_NLS 21   /* line-search evaluations, same */
#define TSG_INFO_BARFORCE 22
#define TSG_INFO_MAXCFRC 23
#define TSG_INFO_WAYPT 24
#define TSG_INFO_ORI 26
#define TSG_INFO_OVERFLOW 28
#define TSG_INFO_BAD 29
#define TSG_INFO_NMPR 30
#define TSG_INFO_RESET_PSI 31 /* heading at the last reset (reward direction of `straight`) */

const char *tsg_last_error(void);
int tsg_version(void);
int tsg_device_count(void);

/* n_envs independent envs on CUDA device `device`; env_id_base offsets the RNG stream ids (rank sharding).
 * Replaces MujocoEnv.__init__ -> MjModel.from_xml_path + MjData (tr_env.py:274-276, tensegrity_env.py:239-241) and the
 * env constructor's bookkeeping (tr_env.py:130-285). */
int tsg_create(const TsgModel *model, const TsgEnvConfig *cfg, int n_envs, int device, long long env_id_base,
               TsgHandle **out);
/* same, with n_pool background reset slots: every tsg_step(auto_reset=1) launch also advances each not-yet-ready
 * slot by one of the reset's 50 warm-up env steps, and envs that are done receive a ready slot (state, heading ring,
 * reset observation) instead of resetting synchronously -- the 1000-substep reset latency leaves the step path.
 * Done envs that find no ready slot fall back to the synchronous reset.  tsg_reset(mask = NULL) prewarms all slots. */
int tsg_create_pooled(const TsgModel *model, const TsgEnvConfig *cfg, int n_envs, int n_pool, int device,
                      long long env_id_base, TsgHandle **out);
/* same, choosing the arithmetic of the physics kernels (TSG_PRECISION_*) */
int tsg_create_opts(const TsgModel *model, const TsgEnvConfig *cfg, int n_envs, int n_pool, int device,
                    long long env_id_base, int precision, TsgHandle **out);
int tsg_precision(const TsgHandle *h);
/* counts3 = {done envs, ready slots, slots handed out} of the last auto-reset (synchronous read) */
int tsg_pool_stats_host(TsgHandle *h, int *counts3);
int tsg_destroy(TsgHandle *h);
int tsg_num_envs(const TsgHandle *h);
int tsg_obs_dim(const TsgHandle *h);
int tsg_launches(const TsgHandle *h); /* kernels launched so far by this handle */
/* step-kernel launch shape of this handle (for occupancy reports): *warps_per_cta = warps per CTA * 100 + lanes per
 * env (603 = 6 warps, 3 lanes per env), dynamic shared memory per CTA, registers per thread */
int tsg_kernel_config(const TsgHandle *h, int *warps_per_cta, int *smem_bytes, int *regs_per_thread);

/* Replaces env.reset(): MujocoEnv.reset -> reset_model (tr_env.py:709-872, tensegrity_env.py:433-512; run.py:119).
 * reset the envs whose mask byte is non-zero (mask_dev NULL = all).  draws_in_dev: optional
 * [n_envs][TSG_NDRAW] explicit random draws (tests); otherwise Philox(seed, env id, reset count).
 * obs_dev / obs32_dev (optional) receive the reset observation rows of the reset envs;
 * term_obs_dev (optional) first receives a copy of obs_dev rows about to be overwritten. */
int tsg_reset(TsgHandle *h, const uint8_t *mask_dev, unsigned long long seed, const double *draws_in_dev,
              double *obs_dev, float *obs32_dev, double *term_obs_dev, void *stream);

/* Replaces env.step(action): tr_env.step (tr_env.py:327-527) / tensegrity_env.step (tensegrity_env.py:291-410),
 * i.e. do_simulation -> mujoco.mj_step(nstep = frame_skip) + mj_rnePostConstraint, _get_obs, reward, termination
 * (run.py:138).  info columns = the reference's info dict keys (TSG_INFO_*; tr_env.py:496-512).
 * one env step for all envs.  ctrl_dev: [n_envs][6] (f64 or f32 per ctrl_dtype).  Optional outputs:
 * obs_dev [n][obs_dim] f64, obs32_dev f32 copy, reward_dev [n] f64, done_dev [n] u8
 * (terminated|truncated), info_dev [n][TSG_INFO_DIM] f64.  If auto_reset != 0 the envs that are done
 * are reset in the same call (their obs rows then hold the first observation of the new episode
 * and term_obs_dev, if given, the terminal one). */
int tsg_step(TsgHandle *h, const void *ctrl_dev, int ctrl_dtype, double *obs_dev, float *obs32_dev,
             double *reward_dev, uint8_t *done_dev, double *info_dev, int auto_reset, unsigned long long seed,
             double *term_obs_dev, void *stream);

/* Observation noise (TsgEnvConfig.use_obs_noise; tr_env.py:524-527): tsg_step / tsg_reset then return the NOISY
 * observation, as the reference does.  real_obs_dev (optional, [n_envs][obs_dim] f64, device) additionally receives
 * the noise-free observation of every step -- the reference's info["real_observation"] (tr_env.py:505).  The
 * normal draws are Philox(seed, env id, reset count, episode step): reproducible, unlike the reference's unseeded
 * np.random.default_rng() (tr_env.py:552).  The handle owns a default buffer (read it with tsg_get_real_obs_host);
 * pass a device buffer to have the rows written there instead (it must outlive the calls), NULL to switch back. */
int tsg_set_real_obs(TsgHandle *h, double *real_obs_dev);
/* the noise-free observations of the last step / reset, HOST buffer [n_envs][obs_dim] (synchronous) */
int tsg_get_real_obs_host(TsgHandle *h, double *real_obs);

/* mj_forward on the stored states (MujocoEnv.set_state -> mujoco.mj_forward; tr_env.py:744,763,800):
 * refreshes the kinematics-derived bookkeeping, optional obs/info */
int tsg_forward(TsgHandle *h, double *obs_dev, double *info_dev, void *stream);

/* same from host code (MujocoEnv.set_state of a single env): runs on the handle's own stream -- ordered with
 * tsg_step_host / tsg_reset_host -- and returns after the optional HOST obs / info rows are written */
int tsg_forward_host(TsgHandle *h, double *obs, double *info);

/* raw state access (HOST buffers, synchronous): any pointer may be NULL.  Replaces reads / writes of data.qpos,
 * data.qvel, data.act, data.qacc_warmstart, data.ctrl (tr_env.py:345,583; MujocoEnv.set_state) */
int tsg_get_state_host(TsgHandle *h, double *qpos, double *qvel, double *act, double *qacc_warmstart, double *ctrl);
int tsg_set_state_host(TsgHandle *h, const double *qpos, const double *qvel, const double *act,
                       const double *qacc_warmstart, const double *ctrl);
/* whole records [n_envs][TSG_STATE_STRIDE] (checkpoint / restore of env state), HOST buffers */
int tsg_get_records_host(TsgHandle *h, double *records);
int tsg_set_records_host(TsgHandle *h, const double *records);
/* the heading rings [n_envs][TSG_HEADING_SLOTS] that the records' cursors index (turn / aiming reward delay):
 * a checkpoint of env state is records + heading rings */
int tsg_get_heading_host(TsgHandle *h, double *heading);
int tsg_set_heading_host(TsgHandle *h, const double *heading);
/* last reset draws [n_envs][TSG_NDRAW], HOST buffer */
int tsg_get_draws_host(TsgHandle *h, double *draws);

/* Per-env tendon and actuator parameters (domain randomisation, system identification).  Every env record and every
 * pool slot has a row of TSG_NPARAM doubles (TSG_PARAM_*) that replaces the model's ten_stiffness, ten_damping,
 * ten_lengthspring, act_gain, act_bias and act_dynprm0 for that env.  Until one of the two setters is called a handle
 * runs the model's constants; the first call gives every row the nominal row and switches the handle to the per-env
 * kernels for good.
 *
 * tsg_set_param_ranges: HOST arrays lo, hi [TSG_NPARAM] of scale factors.  From then on every reset (tsg_reset, the
 * synchronous auto-reset of tsg_step, and a pool slot's restart) draws a new row nominal[i] * U(lo[i], hi[i]).  The
 * draws are Philox(seed ^ key, stream, (reset count << 8) | k) with the stream ids of the reset draws (env id, or
 * 2^40 + slot id), so sharded handles reproduce an unsharded one.  Rules: finite, 0 <= lo <= hi, an act_dynprm0
 * scale above 0; the lower and upper lengthspring of a tendon share one draw and need equal ranges.  lo = hi = NULL
 * stops the draws (rows then stay as they are at resets).  Synchronises the device.
 *
 * tsg_set_env_params: explicit rows [n_envs][TSG_NPARAM] (DEVICE) for the envs whose mask byte is non-zero (NULL =
 * all), in effect from the next launch on the stream; with ranges set they last until the env's next reset.  Fails on
 * a handle with a reset pool: an env that receives a pool slot takes the row the slot was warmed up with.
 *
 * tsg_get_env_params: every env's row [n_envs][TSG_NPARAM] (DEVICE).  A checkpoint of env state is records + heading
 * rings + parameter rows. */
int tsg_set_param_ranges(TsgHandle *h, const double *lo, const double *hi);
int tsg_set_env_params(TsgHandle *h, const double *params_dev, const uint8_t *mask_dev, void *stream);
int tsg_get_env_params(TsgHandle *h, double *params_dev, void *stream);

/* the calls behind the reference-shaped single env (envs.py tr_env / tensegrity_env: run.py:119,138): host buffers
 * in, host buffers out,
 * H2D/D2H copies on the handle's stream, synchronous. */
int tsg_step_host(TsgHandle *h, const double *ctrl, double *obs, double *reward, uint8_t *done, double *info,
                  int auto_reset, unsigned long long seed, double *term_obs);
int tsg_reset_host(TsgHandle *h, const uint8_t *mask, unsigned long long seed, const double *draws_in, double *obs);

#ifdef __cplusplus
}
#endif
#endif /* TSG_H_ */
