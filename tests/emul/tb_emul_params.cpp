// tb_emul_params.cpp -- TEST HARNESS ONLY.  The fibre-warp emulator of tb_emul.cpp (included whole: same runtime, same
// tbe_* entry points) plus the per-env-parameter variant of the kernel source, tb_env_kernel<PerEnv<P>, ...>'s device
// code.  A tbp handle rides on a tbe handle (model, env config, noise keys) and owns the per-env variant's env slices;
// the caller owns the parameter rows [n_envs (+ n_pool)][NPARAM] and the {nominal, lo, hi}[NPARAM] ranges of the reset
// draws, as the device library owns d_params / d_prange.  Used by tests/test_env_params.py and, for the expected
// draws, tests/test_gpu_env_params.py.
#include "tb_emul.cpp"

struct EmulP {
  Emul* E;
  EnvSh<PerEnv<P64>> S[EPW];
  EnvSh<PerEnv<P32>> SF[EPW];
  Con<double> spill[EPW][3 * KS];
  Con<double> spillf[EPW][3 * KS];
  double* params; const double* prange;
};

template <typename F> static void run_p(EmulP* P, F body) {
  run_warp([&]() { LaneCtx L = make_lane(); body(P->S[L.grp], L); });
}
static StepIO make_io_p(const EmulP* P, int n, double* rec, double* heading) {
  StepIO io = make_io(n, rec, heading, P->E);
  io.params = P->params; io.prange = P->prange;
  return io;
}

// raw physics as tbe_mj_step / tbe_mj_step_f32, each env with its row
template <typename PR>
static void mj_step_p(EmulP* P, EnvSh<PR>* slices, const ModelT<typename PR::real>& m, int n, double* rec,
                      const double* ctrl, int nstep, double* ten_length, double* cfrc_ext, int* stats) {
  const StepIO io = make_io_p(P, n, rec, nullptr);
  run_warp([&]() {
    LaneCtx L = make_lane();
    EnvSh<PR>& S = slices[L.grp];
    const bool on = L.valid && L.grp < n;
    Aux A;
    double head[HEADING_SLOTS];
    double* r = rec + (size_t)(on ? L.grp : 0) * STATE_STRIDE;
    load_env(S, L, on, A, r, head);
    if (on && L.bar == 0) { for (int i = 0; i < NACT; i++) S.ctrl[i] = ctrl[(size_t)L.grp * NACT + i]; set_prm_row(S, io, (size_t)L.grp); }
    wsync();
    simulate(S, m, L, on, nstep, true, false);
    if (on && L.bar == 0) {
      int e = L.grp;
      if (ten_length) for (int i = 0; i < NTEN; i++) ten_length[e * NTEN + i] = S.tlen[i];
      if (cfrc_ext) for (int i = 0; i < 24; i++) cfrc_ext[e * 24 + i] = S.cfrc[i];
      if (stats) { int* s = stats + 6 * e; s[0] = S.nact; s[1] = S.niter; s[2] = S.nls; s[3] = S.nmpr; s[4] = S.overflow; s[5] = S.bad; }
    }
    wsync();
    store_env(S, L, on, A, r);
  });
}
extern "C" {

// the per-env variant on tbe handle `h`: rows (kept and updated in place), prange (NULL = rows kept at resets)
void* tbp_create(void* h, double* rows, const double* prange) {
  EmulP* P = new EmulP();
  memset(P->S, 0, sizeof(P->S));
  memset(P->SF, 0, sizeof(P->SF));
  for (int g = 0; g < EPW; g++) { P->S[g].spill = P->spill[g]; P->SF[g].spill = P->spillf[g]; }
  P->E = (Emul*)h; P->params = rows; P->prange = prange;
  return P;
}
void tbp_destroy(void* p) { delete (EmulP*)p; }

void tbp_step(void* p, int n, double* rec, double* heading, const double* ctrl, double* obs, double* reward,
              uint8_t* done, double* info) {
  EmulP* P = (EmulP*)p;
  StepIO io = make_io_p(P, n, rec, heading);
  io.ctrl64 = ctrl; io.obs = obs; io.reward = reward; io.done = done; io.info = info;
  run_p(P, [&](EnvSh<PerEnv<P64>>& S, const LaneCtx& L) { run_step(S, P->E->m, P->E->c, io, L, 0, false); });
}
void tbp_reset(void* p, int n, double* rec, double* heading, double* draws, int explicit_draws, unsigned long long seed,
               long long env_id, double* obs, const uint8_t* mask) {
  EmulP* P = (EmulP*)p;
  P->E->seed = seed; P->E->env_id = env_id;
  StepIO io = make_io_p(P, n, rec, heading);
  io.draws = draws; io.explicit_draws = explicit_draws; io.obs = obs; io.mask = mask;
  run_p(P, [&](EnvSh<PerEnv<P64>>& S, const LaneCtx& L) { run_reset(S, P->E->m, P->E->c, io, L, 0); });
}
void tbp_forward(void* p, int n, double* rec, double* heading, double* obs, double* info) {
  EmulP* P = (EmulP*)p;
  StepIO io = make_io_p(P, n, rec, heading);
  io.obs = obs; io.info = info;
  run_p(P, [&](EnvSh<PerEnv<P64>>& S, const LaneCtx& L) { run_forward(S, P->E->m, P->E->c, io, L, 0); });
}
void tbp_pool(void* p, int n_envs, int n_pool, double* rec, double* heading, double* draws, double* pool_obs,
              unsigned long long seed, int finish_now) {
  EmulP* P = (EmulP*)p;
  P->E->seed = seed;
  StepIO io = make_io_p(P, n_envs, rec, heading);
  io.n_pool = n_pool; io.draws = draws; io.pool_obs = pool_obs;
  run_p(P, [&](EnvSh<PerEnv<P64>>& S, const LaneCtx& L) { run_pool(S, P->E->m, P->E->c, io, L, 0, finish_now != 0); });
}
void tbp_mj_step(void* p, int n, double* rec, const double* ctrl, int nstep, double* ten_length, double* cfrc_ext, int* stats) {
  EmulP* P = (EmulP*)p;
  mj_step_p(P, P->S, P->E->m, n, rec, ctrl, nstep, ten_length, cfrc_ext, stats);
}
void tbp_mj_step_f32(void* p, int n, double* rec, const double* ctrl, int nstep, double* ten_length, int* stats) {
  EmulP* P = (EmulP*)p;
  mj_step_p(P, P->SF, P->E->f32->m, n, rec, ctrl, nstep, ten_length, nullptr, stats);
}
// the rows one reset draws: n rows for streams stream0 .. stream0 + n - 1
void tbp_param_draws(double* out, const double* prange, unsigned long long seed, unsigned long long stream0,
                     unsigned long long nreset, int n) {
  for (int k = 0; k < n; k++) draw_params(out + (size_t)k * NPARAM, prange, seed, stream0 + k, nreset);
}
void tbp_nominal_params(const TsgModel* model, double* row) { nominal_params(*model, row); }
}
