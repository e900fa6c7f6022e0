// tb_emul.cpp -- TEST HARNESS ONLY.  Compiles the device source of the bar-lane kernel (csrc/tb_*.cuh) as plain C++
// with TB_EMUL and runs ONE WARP of it on the CPU: the 32 lanes are cooperative fibres (ucontext), and the SIMT
// primitives of tb_simt.h (shuffle, ballot, warp barrier) are rendezvous points between them.  Lane-private code runs
// serially lane by lane between two rendezvous, so races across lanes, missing barriers and non-uniform control flow
// at an exchange point show up here (deadlock detection aborts) without a GPU.  Both variants of the env kernels run
// here: the default one and the per-env-parameter one, tb_env_kernel<PerEnv<P>, ...>'s device code.  Used by
// tests/test_emul_vs_oracle.py and tests/test_env_params.py to check the CUDA source against the oracle, and by
// tests/test_gpu_env_params.py for the expected parameter draws.  Not part of libtsg.so, never reachable from the
// product package.
#define TB_EMUL 1
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ucontext.h>

#include <functional>
#include <string>
#include <tuple>

#include "../../tensegrity_rl_b200/csrc/tb_env.cuh"

namespace tb {
// ------------------------------------------------------------------ fibre warp
static constexpr int NL = 32;
static ucontext_t g_main, g_ctx[NL];
static char* g_stack[NL];
static bool g_done[NL];
static int g_cur = 0;
static unsigned g_gen = 0;
static int g_arrived = 0;
static unsigned long g_progress = 0;
static uint64_t g_xbuf[NL];
static bool g_pbuf[NL];
static std::function<void()> g_body;

int emu_lane() { return g_cur; }
static void yield_() { swapcontext(&g_ctx[g_cur], &g_main); }
void emu_sync() {
  unsigned g = g_gen;
  if (++g_arrived == NL) { g_arrived = 0; g_gen++; g_progress++; return; }
  while (g_gen == g) yield_();
}
uint64_t emu_shfl(uint64_t bits, int src) {
  g_xbuf[g_cur] = bits;
  emu_sync();
  uint64_t r = g_xbuf[src & (NL - 1)];
  emu_sync();
  return r;
}
unsigned emu_ballot(bool p) {
  g_pbuf[g_cur] = p;
  emu_sync();
  unsigned r = 0;
  for (int i = 0; i < NL; i++) if (g_pbuf[i]) r |= 1u << i;
  emu_sync();
  return r;
}
static void trampoline() {
  g_body();
  g_done[g_cur] = true;
  g_progress++;
  swapcontext(&g_ctx[g_cur], &g_main);
}
static void run_warp(std::function<void()> body) {
  static const size_t STK = 1 << 20;
  g_body = body;
  g_arrived = 0;
  for (int i = 0; i < NL; i++) {
    if (!g_stack[i]) g_stack[i] = (char*)malloc(STK);
    getcontext(&g_ctx[i]);
    g_ctx[i].uc_stack.ss_sp = g_stack[i];
    g_ctx[i].uc_stack.ss_size = STK;
    g_ctx[i].uc_link = &g_main;
    makecontext(&g_ctx[i], trampoline, 0);
    g_done[i] = false;
  }
  for (;;) {
    unsigned long before = g_progress;
    bool all = true;
    for (int i = 0; i < NL; i++) {
      if (g_done[i]) continue;
      all = false;
      g_cur = i;
      swapcontext(&g_main, &g_ctx[i]);
    }
    if (all) break;
    if (g_progress == before) {
      fprintf(stderr, "tb_emul: warp deadlock (%d lanes at a barrier, others finished or diverged)\n", g_arrived);
      abort();
    }
  }
}
}  // namespace tb

using namespace tb;

template <typename PR> struct Slices {   // one variant's env slices, each with its contact spill area
  EnvSh<PR> S[EPW];
  Con<typename PR::sreal> spill[EPW][3 * KS];
  Slices() { memset(S, 0, sizeof(S)); for (int g = 0; g < EPW; g++) S[g].spill = spill[g]; }
};
struct Emul {
  ModelT<double> m;
  ModelT<float> mf;   // fp32 physics twin (raw mj_step only: numerics studies of the optional fp32 mode)
  EnvCfg c;
  float* hdata;
  std::tuple<Slices<P64>, Slices<P32>, Slices<PerEnv<P64>>, Slices<PerEnv<P32>>> slices;
  // the per-env variant runs when params is set (tbe_set_params): the caller's rows [n (+ n_pool)][NPARAM], kept and
  // updated in place as the device library keeps d_params, and the {nominal, lo, hi}[NPARAM] ranges of the reset draws
  // (null = rows kept at resets)
  double* params; const double* prange;
  unsigned long long seed; long long env_id; double* real_obs;
};

// one warp over the env slices of precision P: the per-env variant's with parameter rows, the default variant's without
template <typename P, typename F> static void on_warp(Emul* E, F body) {
  if (E->params) run_warp([&]() { LaneCtx L = make_lane(); body(std::get<Slices<PerEnv<P>>>(E->slices).S[L.grp], L); });
  else run_warp([&]() { LaneCtx L = make_lane(); body(std::get<Slices<P>>(E->slices).S[L.grp], L); });
}
static StepIO make_io(int n, double* rec, double* heading, const Emul* E) {
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.state = rec; io.heading = heading; io.n_envs = n;
  io.seed = E->seed; io.env_id_base = E->env_id; io.real_obs = E->real_obs;
  io.params = E->params; io.prange = E->prange;
  return io;
}
// raw physics: nstep x mj_step on the records with the given ctrl (no env semantics), then cfrc_ext
template <typename P>
static void mj_step(Emul* E, const ModelT<typename P::real>& m, int n, double* rec, const double* ctrl, int nstep,
                    double* ten_length, double* cfrc_ext, int* stats) {
  const StepIO io = make_io(n, rec, nullptr, E);
  on_warp<P>(E, [&](auto& S, const LaneCtx& L) {
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

const char* tbe_create(const TsgModel* model, const TsgEnvConfig* cfg, void** out) {
  static std::string err;
  Emul* E = new Emul();
  if (model->floor_type == TSG_FLOOR_HFIELD) {
    size_t n = (size_t)model->hf_nrow * model->hf_ncol;
    E->hdata = (float*)malloc(n * sizeof(float));
    memcpy(E->hdata, model->hf_data, n * sizeof(float));
  }
  err = make_model<double>(*model, E->m, E->hdata);
  if (err.empty()) err = make_model<float>(*model, E->mf, E->hdata);
  if (err.empty()) err = make_env_cfg(*cfg, *model, E->c);
  if (!err.empty()) { free(E->hdata); delete E; return err.c_str(); }
  *out = E;
  return nullptr;
}
void tbe_destroy(void* h) { Emul* E = (Emul*)h; free(E->hdata); delete E; }
int tbe_envs_per_warp() { return EPW; }

// rows = null: the default variant from now on
void tbe_set_params(void* h, double* rows, const double* prange) {
  Emul* E = (Emul*)h; E->params = rows; E->prange = prange;
}
void tbe_set_noise(void* h, unsigned long long seed, long long env_id, double* real_obs) {
  Emul* E = (Emul*)h; E->seed = seed; E->env_id = env_id; E->real_obs = real_obs;
}
void tbe_obs_normals(unsigned long long seed, unsigned long long stream, unsigned long long nreset,
                     unsigned long long step, int n, double* out) {
  for (int pr = 0; pr < (n + 1) / 2; pr++) {
    double z0, z1;
    noise_pair(seed, stream, nreset, step, pr, z0, z1);
    out[2 * pr] = z0;
    if (2 * pr + 1 < n) out[2 * pr + 1] = z1;
  }
}
// n <= EPW envs, records [n][96], heading [n][32], ctrl [n][6]; outputs per env
void tbe_step(void* h, int n, double* rec, double* heading, const double* ctrl, double* obs, double* reward,
              uint8_t* done, double* info) {
  Emul* E = (Emul*)h;
  StepIO io = make_io(n, rec, heading, E);
  io.ctrl64 = ctrl; io.obs = obs; io.reward = reward; io.done = done; io.info = info;
  on_warp<P64>(E, [&](auto& S, const LaneCtx& L) { run_step(S, E->m, E->c, io, L, 0, false); });
}
void tbe_reset(void* h, int n, double* rec, double* heading, double* draws, int explicit_draws, unsigned long long seed,
               long long env_id, double* obs, const uint8_t* mask) {
  Emul* E = (Emul*)h;
  E->seed = seed; E->env_id = env_id;
  StepIO io = make_io(n, rec, heading, E);
  io.draws = draws; io.explicit_draws = explicit_draws; io.obs = obs; io.mask = mask;
  on_warp<P64>(E, [&](auto& S, const LaneCtx& L) { run_reset(S, E->m, E->c, io, L, 0); });
}
void tbe_forward(void* h, int n, double* rec, double* heading, double* obs, double* info) {
  Emul* E = (Emul*)h;
  StepIO io = make_io(n, rec, heading, E);
  io.obs = obs; io.info = info;
  on_warp<P64>(E, [&](auto& S, const LaneCtx& L) { run_forward(S, E->m, E->c, io, L, 0); });
}
// background pool: n_envs records followed by n_pool slot records; advances every slot by one launch
void tbe_pool(void* h, int n_envs, int n_pool, double* rec, double* heading, double* draws, double* pool_obs,
              unsigned long long seed, int finish_now) {
  Emul* E = (Emul*)h;
  E->seed = seed;
  StepIO io = make_io(n_envs, rec, heading, E);
  io.n_pool = n_pool; io.draws = draws; io.pool_obs = pool_obs;
  on_warp<P64>(E, [&](auto& S, const LaneCtx& L) { run_pool(S, E->m, E->c, io, L, 0, finish_now != 0); });
}
void tbe_mj_step(void* h, int n, double* rec, const double* ctrl, int nstep, double* ten_length, double* cfrc_ext,
                 int* stats) {
  Emul* E = (Emul*)h;
  mj_step<P64>(E, E->m, n, rec, ctrl, nstep, ten_length, cfrc_ext, stats);
}
void tbe_mj_step_f32(void* h, int n, double* rec, const double* ctrl, int nstep, double* ten_length, int* stats) {
  Emul* E = (Emul*)h;
  mj_step<P32>(E, E->mf, n, rec, ctrl, nstep, ten_length, nullptr, stats);
}
void tbe_reset_noise(unsigned long long seed, unsigned long long stream, unsigned long long nreset, double* out39) {
  for (int i = 0; i < NQ + NV; i++) out39[i] = reset_noise_draw(seed, stream, nreset, i);
}
void tbe_make_draws(double* d, unsigned long long seed, unsigned long long env_id, unsigned long long nreset) {
  make_draws(d, seed, env_id, nreset);
}
// the parameter rows one reset draws: n rows for streams stream0 .. stream0 + n - 1
void tbe_param_draws(double* out, const double* prange, unsigned long long seed, unsigned long long stream0,
                     unsigned long long nreset, int n) {
  for (int k = 0; k < n; k++) draw_params(out + (size_t)k * NPARAM, prange, seed, stream0 + k, nreset);
}
void tbe_nominal_params(const TsgModel* model, double* row) { nominal_params(*model, row); }
}
