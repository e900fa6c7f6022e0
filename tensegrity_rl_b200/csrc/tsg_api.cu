// tsg_api.cu -- kernels and the C ABI (include/tsg.h) of libtsg.so.  sm_100a only.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <string>
#include <vector>

#include "../../include/tsg.h"
#include "tb_env.cuh"

using namespace tb;

// Production configuration (profiles/): three lanes per env, ten envs per warp, TB_WARPS warps per CTA and
// TB_MIN_CTAS CTAs per SM (the register cap follows: 65536 / (TB_MIN_CTAS * TB_WARPS * 32) per thread).  The step
// kernel runs its warps aligned: the warps of a CTA walk through an env step in phase (CTA barriers at every substep
// and Newton iteration), so that they share fetched instructions.
#ifndef TB_MIN_CTAS
#define TB_MIN_CTAS 1
#endif
#ifndef TB_WARPS
#define TB_WARPS 6   // 60 envs x 3664 B + model = 224 080 B of the 227 KB: the most that fits (5 warps: -3.5 %, 4: -17 %)
#endif
#ifndef TB_WARPS_SMALL
#define TB_WARPS_SMALL 2   // second CTA shape of the step kernel (two CTAs per SM), for batches that fit the machine at once
#endif
#ifndef TB_EPW_SMALL
#define TB_EPW_SMALL 10    // envs per warp in that shape (fewer envs per warp = fewer envs waiting for the slowest one)
#endif

static_assert(STATE_STRIDE == TSG_STATE_STRIDE && INFO_DIM == TSG_INFO_DIM && NDRAW == TSG_NDRAW, "ABI constants");
static_assert(SO_USED <= STATE_STRIDE, "state record too small");
static_assert(HEADING_SLOTS == TSG_HEADING_SLOTS, "heading slots");
static_assert(NPARAM == TSG_NPARAM && PRM_TK == TSG_PARAM_TEN_STIFFNESS && PRM_TDAMP == TSG_PARAM_TEN_DAMPING &&
              PRM_TLS == TSG_PARAM_TEN_LENGTHSPRING && PRM_GAIN == TSG_PARAM_ACT_GAIN && PRM_BIAS == TSG_PARAM_ACT_BIAS &&
              PRM_DYNPRM0 == TSG_PARAM_ACT_DYNPRM0, "param row layout");

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_FORWARD = 2 };

__host__ __device__ constexpr size_t align16(size_t x) { return (x + 15) & ~size_t(15); }
template <typename P> __host__ __device__ constexpr size_t smem_model() { return align16(sizeof(ModelT<typename P::real>)); }
constexpr size_t SMEM_CFG = align16(sizeof(EnvCfg));
// env slices are spaced by an odd number of 16-byte units, so that the same field of the ten envs of a warp falls into different banks
template <typename P> __host__ __device__ constexpr size_t envsh_stride() { return align16(sizeof(EnvSh<P>)) | 16; }
template <typename P, int W, int E = EPW> constexpr size_t smem_bytes() { return smem_model<P>() + SMEM_CFG + (size_t)W * E * envsh_stride<P>(); }

// Persistent CTAs: the grid fills the machine once (SMs x resident CTAs) and every CTA pulls rounds of TB_WARPS chunks
// (a chunk = EPW consecutive envs, or pool slots, stepped by one warp) from a global counter until the batch is done,
// so rounds of different cost (contact count, Newton iterations, resets) balance dynamically.  The env rounds come
// first, then the pool rounds, so that all warps of a CTA always run the same program.  The model constants are
// staged once per CTA in shared memory.
template <typename P, int MODE, int W, int E = EPW>
__global__ void __launch_bounds__(W * 32, TB_MIN_CTAS) tb_env_kernel(const ModelT<typename P::real>* __restrict__ gm,
                                                                            const EnvCfg* __restrict__ gc, StepIO io,
                                                                            Con<typename P::sreal>* __restrict__ spill_base) {
  typedef typename P::real real;
  extern __shared__ __align__(16) unsigned char tb_smem[];
  __shared__ int s_round;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(gm);
    uint32_t* dst = reinterpret_cast<uint32_t*>(tb_smem);
    for (int i = threadIdx.x; i < (int)(sizeof(ModelT<real>) / 4); i += blockDim.x) dst[i] = src[i];
    src = reinterpret_cast<const uint32_t*>(gc);
    dst = reinterpret_cast<uint32_t*>(tb_smem + smem_model<P>());
    for (int i = threadIdx.x; i < (int)(sizeof(EnvCfg) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const ModelT<real>& m = *reinterpret_cast<const ModelT<real>*>(tb_smem);
  const EnvCfg& c = *reinterpret_cast<const EnvCfg*>(tb_smem + smem_model<P>());
  const LaneCtx L = make_lane(E);
  const int warp = threadIdx.x >> 5;
  EnvSh<P>& S = *reinterpret_cast<EnvSh<P>*>(tb_smem + smem_model<P>() + SMEM_CFG +
                                                   (size_t)(warp * E + L.grp) * envsh_stride<P>());
  if (L.valid && L.bar == 0) S.spill = spill_base + (size_t)((blockIdx.x * W + warp) * EPW + L.grp) * (3 * KS);
  __syncwarp();
  const int env_chunks = (io.n_envs + E - 1) / E, env_rounds = (env_chunks + W - 1) / W;
  const int pool_chunks = (MODE == MODE_STEP || (MODE == MODE_RESET && !io.mask)) ? (io.n_pool + E - 1) / E : 0;
  const int pool_rounds = (pool_chunks + W - 1) / W;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_round = atomicAdd(io.counter, 1);
    __syncthreads();
    const int round = s_round;
    if (round >= env_rounds + pool_rounds) break;
    if (round < env_rounds) {
      const int first = (round * W + warp) * E;   // may lie beyond the batch: the warp then idles in step
      if (MODE == MODE_STEP) run_step(S, m, c, io, L, first, true);
      else if (MODE == MODE_RESET) run_reset(S, m, c, io, L, first);
      else run_forward(S, m, c, io, L, first);
    } else run_pool(S, m, c, io, L, ((round - env_rounds) * W + warp) * E, MODE == MODE_RESET);
  }
}

// Hand ready pool slots to envs that are done (one CTA; ordered, hence deterministic: the k-th done env gets the
// k-th ready slot).  Copies record (all but the env's own reset counter, which is incremented), heading ring and reset observation;
// the slot restarts from phase 0 with its next draw.  Done envs left without a slot are flagged in need_sync.
__global__ void __launch_bounds__(1024) tsg_assign_kernel(double* __restrict__ state, double* __restrict__ heading,
                                                           const uint8_t* __restrict__ done, uint8_t* __restrict__ need_sync,
                                                           double* obs, float* obs32, double* term_obs,
                                                           const double* __restrict__ pool_obs, const double* __restrict__ pool_real_obs, double* real_obs, int* __restrict__ lists,
                                                           int* __restrict__ counts, int n, int n_pool, int obs_dim, int ready_phase) {
  __shared__ int wcount[32], woff[32], s_ndone, s_nready;
  int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int* done_list = lists;            // first n_pool done envs, in env order
  int* ready_list = lists + n_pool;  // ready pool slots, in slot order
  for (int pass = 0; pass < 2; pass++) {  // pass 0: done envs, pass 1: ready slots
    int total = pass == 0 ? n : n_pool;
    int seg = ((total + 31) / 32 + 31) / 32 * 32, lo = warp * seg, hi = min(total, lo + seg);
    int cnt = 0;
    for (int b = lo; b < hi; b += 32) {
      int i = b + lane;
      bool f = i < hi && (pass == 0 ? done[i] != 0 : (int)state[(size_t)(n + i) * STATE_STRIDE + SO_FLAGS] == ready_phase);
      cnt += __popc(__ballot_sync(0xffffffffu, f));
    }
    if (lane == 0) wcount[warp] = cnt;
    __syncthreads();
    if (tid == 0) { int s = 0; for (int w = 0; w < 32; w++) { woff[w] = s; s += wcount[w]; } if (pass == 0) s_ndone = s; else s_nready = s; }
    __syncthreads();
    int off = woff[warp];
    int* out = pass == 0 ? done_list : ready_list;
    for (int b = lo; b < hi; b += 32) {
      int i = b + lane;
      bool f = i < hi && (pass == 0 ? done[i] != 0 : (int)state[(size_t)(n + i) * STATE_STRIDE + SO_FLAGS] == ready_phase);
      unsigned mk = __ballot_sync(0xffffffffu, f);
      int k = off + __popc(mk & ((1u << lane) - 1));
      if (f && k < n_pool) out[k] = i;
      off += __popc(mk);
    }
    __syncthreads();
  }
  int npair = min(min(s_ndone, s_nready), n_pool);
  if (tid == 0) { counts[0] = s_ndone; counts[1] = s_nready; counts[2] = npair; }
  if (need_sync) for (int i = tid; i < n; i += blockDim.x) need_sync[i] = done[i];
  __syncthreads();
  for (int k = warp; k < npair; k += 32) {
    int e = done_list[k], p = ready_list[k];
    double* dst = state + (size_t)e * STATE_STRIDE;
    double* src = state + (size_t)(n + p) * STATE_STRIDE;
    for (int i = lane; i < STATE_STRIDE; i += 32) if (i != SO_NRESET && i != SO_FLAGS) dst[i] = src[i];
    for (int i = lane; i < HEADING_SLOTS; i += 32) heading[(size_t)e * HEADING_SLOTS + i] = heading[(size_t)(n + p) * HEADING_SLOTS + i];
    for (int i = lane; i < obs_dim; i += 32) {
      double v = pool_obs[(size_t)p * obs_dim + i];
      if (obs) { if (term_obs) term_obs[(size_t)e * obs_dim + i] = obs[(size_t)e * obs_dim + i]; obs[(size_t)e * obs_dim + i] = v; }
      if (obs32) obs32[(size_t)e * obs_dim + i] = (float)v;
      if (real_obs && pool_real_obs) real_obs[(size_t)e * obs_dim + i] = pool_real_obs[(size_t)p * obs_dim + i];
    }
    if (lane == 0) { src[SO_FLAGS] = 0; src[SO_NRESET] += 1; dst[SO_NRESET] += 1; if (need_sync) need_sync[e] = 0; }
  }
}

// record <-> separate arrays (tsg_get_state / tsg_set_state)
__global__ void tsg_gather_kernel(const double* __restrict__ state, int n, double* qpos, double* qvel, double* act,
                                  double* warm, double* ctrl) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const double* r = state + (size_t)e * STATE_STRIDE;
  if (qpos) for (int i = 0; i < NQ; i++) qpos[(size_t)e * NQ + i] = r[SO_QPOS + i];
  if (qvel) for (int i = 0; i < NV; i++) qvel[(size_t)e * NV + i] = r[SO_QVEL + i];
  if (warm) for (int i = 0; i < NV; i++) warm[(size_t)e * NV + i] = r[SO_WARM + i];
  if (ctrl) for (int i = 0; i < NACT; i++) ctrl[(size_t)e * NACT + i] = r[SO_CTRL + i];
  if (act) for (int i = 0; i < NACT; i++) act[(size_t)e * NACT + i] = r[SO_ACT + i];
}
__global__ void tsg_scatter_kernel(double* __restrict__ state, int n, const double* qpos, const double* qvel,
                                   const double* act, const double* warm, const double* ctrl) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  double* r = state + (size_t)e * STATE_STRIDE;
  if (qpos) for (int i = 0; i < NQ; i++) r[SO_QPOS + i] = qpos[(size_t)e * NQ + i];
  if (qvel) for (int i = 0; i < NV; i++) r[SO_QVEL + i] = qvel[(size_t)e * NV + i];
  if (warm) for (int i = 0; i < NV; i++) r[SO_WARM + i] = warm[(size_t)e * NV + i];
  if (ctrl) for (int i = 0; i < NACT; i++) r[SO_CTRL + i] = ctrl[(size_t)e * NACT + i];
  if (act) for (int i = 0; i < NACT; i++) r[SO_ACT + i] = act[(size_t)e * NACT + i];
}
// per-env parameters: the k-th assigned pool slot's row goes to the k-th done env (the pairs tsg_assign_kernel chose)
__global__ void tsg_assign_params_kernel(double* __restrict__ params, const int* __restrict__ lists, const int* __restrict__ counts,
                                         int n, int n_pool) {
  const int npair = counts[2];
  for (int k = blockIdx.x; k < npair; k += gridDim.x) {
    const int e = lists[k], p = lists[n_pool + k];
    for (int i = threadIdx.x; i < NPARAM; i += blockDim.x) params[(size_t)e * NPARAM + i] = params[(size_t)(n + p) * NPARAM + i];
  }
}
// rows [n][NPARAM] = nominal row
__global__ void tsg_fill_params_kernel(double* __restrict__ rows, int n, const double* __restrict__ nominal) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (size_t)n * NPARAM) rows[i] = nominal[i % NPARAM];
}
// rows of the envs whose mask byte is non-zero (mask NULL = all) = src rows
__global__ void tsg_set_params_kernel(double* __restrict__ rows, int n, const double* __restrict__ src, const uint8_t* __restrict__ mask) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (size_t)n * NPARAM && (!mask || mask[i / NPARAM])) rows[i] = src[i];
}
__global__ void tsg_init_records_kernel(double* __restrict__ state, int n, const double* qpos0) {  // n = envs + pool slots
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  double* r = state + (size_t)e * STATE_STRIDE;
  for (int i = 0; i < STATE_STRIDE; i++) r[i] = 0;
  for (int i = 0; i < NQ; i++) r[SO_QPOS + i] = qpos0[i];
}

// ------------------------------------------------------------------ handle
struct TsgHandle {
  int device, n_envs, n_pool, obs_dim, launches, ready_phase, precision;
  long long env_id_base;
  void* d_model; EnvCfg* d_cfg; float* d_hdata; double* d_qpos0;
  double* d_state; double* d_heading; double* d_draws;
  uint8_t* d_done;
  // staging for the host-buffer entry points
  double *d_ctrl, *d_obs, *d_reward, *d_info, *d_termobs, *d_tmp;
  uint8_t* d_mask;
  int* d_counter; void* d_spill;
  double* d_pool_obs; double* d_pool_real_obs; int* d_lists; int* d_counts; uint8_t* d_need_sync;
  double* real_obs;   // where the noise-free observation goes with use_obs_noise: d_realobs_own or the caller's buffer
  double* d_realobs_own;
  // per-env parameters (off until tsg_set_param_ranges / tsg_set_env_params): rows [n_envs + n_pool][NPARAM] and
  // {nominal, lo, hi}[NPARAM] of the reset draws
  double* d_params; double* d_prange;
  int per_env, ranges_on;
  double nominal[NPARAM];
  int grid[3], grid_small, shape, regs, warps, epw;   // shape: 0 = TB_WARPS, 1 = TB_WARPS_SMALL warps per CTA in the step kernel
  int pgrid[3], pgrid_small;   // grids of the per-env kernels
  size_t smem;
  cudaStream_t own_stream;
};

static thread_local std::string g_err;
const char* tsg_last_error(void) { return g_err.c_str(); }
int tsg_version(void) { return 3; }
int tsg_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; } return n; }

#define CK(call)                                                                    \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      g_err = std::string(#call) + ": " + cudaGetErrorString(e_);                   \
      return -2;                                                                    \
    }                                                                               \
  } while (0)
#define FAIL(msg) do { g_err = (msg); return -1; } while (0)

// TSG_EXTRA_SMEM (bytes, env var; measurement aid): pads the dynamic shared memory per CTA to lower the occupancy
static size_t extra_smem() {
  static long v = -1;
  if (v < 0) { const char* e = getenv("TSG_EXTRA_SMEM"); v = e ? atol(e) : 0; }
  return (size_t)v;
}
template <typename P, int MODE, int W, int E = EPW>
static int launch_w(TsgHandle* h, StepIO& io, cudaStream_t s, int counter_slot, int grid) {
  io.counter = h->d_counter + counter_slot;
  tb_env_kernel<P, MODE, W, E><<<grid, W * 32, smem_bytes<P, W, E>() + extra_smem(), s>>>(
      (const ModelT<typename P::real>*)h->d_model, h->d_cfg, io, (Con<typename P::sreal>*)h->d_spill);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}
template <typename P, int MODE>
static int launch_t(TsgHandle* h, StepIO& io, cudaStream_t s, int counter_slot) {
  const int* grid = P::per_env ? h->pgrid : h->grid;
  if (MODE == MODE_STEP && h->shape == 1) return launch_w<P, MODE_STEP, TB_WARPS_SMALL, TB_EPW_SMALL>(h, io, s, counter_slot, P::per_env ? h->pgrid_small : h->grid_small);
  return launch_w<P, MODE, TB_WARPS>(h, io, s, counter_slot, grid[MODE]);
}
// counter_slot: which of the handle's work counters the launch consumes (they are zeroed together, once per API call)
template <int MODE>
static int launch_env(TsgHandle* h, StepIO& io, cudaStream_t s, int counter_slot) {
  const bool f32 = h->precision == TSG_PRECISION_F32;
  if (h->per_env) {
    io.params = h->d_params; io.prange = h->ranges_on ? h->d_prange : nullptr;
    return f32 ? launch_t<PerEnv<P32>, MODE>(h, io, s, counter_slot) : launch_t<PerEnv<P64>, MODE>(h, io, s, counter_slot);
  }
  return f32 ? launch_t<P32, MODE>(h, io, s, counter_slot) : launch_t<P64, MODE>(h, io, s, counter_slot);
}
static int zero_counters(TsgHandle* h, cudaStream_t s) {
  CK(cudaMemsetAsync(h->d_counter, 0, 4 * sizeof(int), s));
  return 0;
}
template <typename P, int MODE, int W, int E = EPW>
static int setup_kernel(TsgHandle* h, int num_sms, int* grid, bool* one_wave = nullptr) {
  size_t smem = smem_bytes<P, W, E>() + extra_smem();
  CK(cudaFuncSetAttribute(tb_env_kernel<P, MODE, W, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tb_env_kernel<P, MODE, W, E>, W * 32, smem));
  if (per_sm < 1) { g_err = "tsg_create: kernel does not fit on an SM"; return -1; }
  // what is not carved out for shared memory stays L1, which serves the spilled contacts and the lanes' local memory
  int need = ((h->n_envs + E - 1) / E + W - 1) / W + ((h->n_pool + E - 1) / E + W - 1) / W;
  int full = num_sms * per_sm;
  *grid = need < full ? need : full;
  if (one_wave) *one_wave = need <= full;
  return 0;
}
template <typename P, int MODE, int W, int E = EPW>
static int note_kernel(TsgHandle* h) {
  cudaFuncAttributes a;
  CK(cudaFuncGetAttributes(&a, tb_env_kernel<P, MODE, W, E>));
  h->regs = a.numRegs; h->smem = smem_bytes<P, W, E>() + extra_smem(); h->warps = W; h->epw = E;
  return 0;
}
// CTA shape of the step kernel.  A batch that fits the machine at once in the small shape (2 CTAs of TB_WARPS_SMALL
// warps per SM) is latency bound by a single round, which is shorter with fewer envs waiting for the slowest one at
// the alignment barriers (4096 envs, steady state: 815k env-steps/s against 740k); larger batches run many rounds per
// SM and the wide shape has the better throughput (131 072 envs: 1.40M against 1.20M).  Fewer envs per warp in the
// small shape (TB_EPW_SMALL 5 or 4 with 3-4 warps) shorten a round only when the machine has room: +8 % at 2048 envs,
// -7 to -14 % at 4096 (more warps per SM, each slower), so the default stays 10.  profiles/r2_ab_variants.log.
static int shape_override() {
  const char* e = getenv("TSG_SHAPE");
  return (e && (e[0] == '0' || e[0] == '1')) ? e[0] - '0' : -1;
}
template <typename P>
static int setup_model(TsgHandle* h, const TsgModel* model, int sms) {
  ModelT<typename P::real> dm;
  std::string err = make_model<typename P::real>(*model, dm, h->d_hdata);
  if (!err.empty()) FAIL("tsg_create: " + err);
  CK(cudaMalloc(&h->d_model, sizeof(dm)));
  CK(cudaMemcpy(h->d_model, &dm, sizeof(dm), cudaMemcpyHostToDevice));
  bool small_one_wave = false;
  if (setup_kernel<P, MODE_STEP, TB_WARPS>(h, sms, &h->grid[MODE_STEP]) ||
      setup_kernel<P, MODE_STEP, TB_WARPS_SMALL, TB_EPW_SMALL>(h, sms, &h->grid_small, &small_one_wave) ||
      setup_kernel<P, MODE_RESET, TB_WARPS>(h, sms, &h->grid[MODE_RESET]) || setup_kernel<P, MODE_FORWARD, TB_WARPS>(h, sms, &h->grid[MODE_FORWARD])) return -2;
  h->shape = shape_override() >= 0 ? shape_override() : (small_one_wave ? 1 : 0);
  if (h->shape == 1 ? note_kernel<P, MODE_STEP, TB_WARPS_SMALL, TB_EPW_SMALL>(h) : note_kernel<P, MODE_STEP, TB_WARPS>(h)) return -2;
  // the per-env kernels (same CTA shapes, a wider env slice) share the contact spill area
  typedef PerEnv<P> PE;
  if (setup_kernel<PE, MODE_STEP, TB_WARPS>(h, sms, &h->pgrid[MODE_STEP]) ||
      setup_kernel<PE, MODE_STEP, TB_WARPS_SMALL, TB_EPW_SMALL>(h, sms, &h->pgrid_small) ||
      setup_kernel<PE, MODE_RESET, TB_WARPS>(h, sms, &h->pgrid[MODE_RESET]) || setup_kernel<PE, MODE_FORWARD, TB_WARPS>(h, sms, &h->pgrid[MODE_FORWARD])) return -2;
  size_t slots = 0;
  for (int k = 0; k < 3; k++) {
    if ((size_t)h->grid[k] * TB_WARPS > slots) slots = (size_t)h->grid[k] * TB_WARPS;
    if ((size_t)h->pgrid[k] * TB_WARPS > slots) slots = (size_t)h->pgrid[k] * TB_WARPS;
  }
  if ((size_t)h->grid_small * TB_WARPS_SMALL > slots) slots = (size_t)h->grid_small * TB_WARPS_SMALL;
  if ((size_t)h->pgrid_small * TB_WARPS_SMALL > slots) slots = (size_t)h->pgrid_small * TB_WARPS_SMALL;
  CK(cudaMalloc(&h->d_spill, slots * EPW * (3 * KS) * sizeof(Con<typename P::sreal>)));   // contact slots beyond the shared-memory pool
  return 0;
}

static int create_impl(TsgHandle* h, const TsgModel* model, const TsgEnvConfig* cfg) {
  const int n_envs = h->n_envs, n_pool = h->n_pool;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, h->device));
  if (prop.major < 10) FAIL("tsg_create: libtsg is built for sm_100a (B200) only");
  if (model->floor_type == TSG_FLOOR_HFIELD) {
    if (!model->hf_data) FAIL("tsg_create: height field data missing");
    size_t nb = (size_t)model->hf_nrow * model->hf_ncol * sizeof(float);
    CK(cudaMalloc(&h->d_hdata, nb));
    CK(cudaMemcpy(h->d_hdata, model->hf_data, nb, cudaMemcpyHostToDevice));
  }
  EnvCfg ec;
  std::string err = make_env_cfg(*cfg, *model, ec);
  if (!err.empty()) FAIL("tsg_create: " + err);
  h->obs_dim = ec.obs_dim; h->ready_phase = ec.warmup_steps + 1;
  nominal_params(*model, h->nominal);
  size_t n = (size_t)n_envs + (size_t)n_pool;
  CK(cudaMalloc(&h->d_cfg, sizeof(EnvCfg)));
  CK(cudaMemcpy(h->d_cfg, &ec, sizeof(ec), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&h->d_qpos0, NQ * sizeof(double)));
  CK(cudaMemcpy(h->d_qpos0, model->qpos0, NQ * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&h->d_state, n * STATE_STRIDE * sizeof(double)));
  CK(cudaMalloc(&h->d_heading, n * HEADING_SLOTS * sizeof(double)));
  CK(cudaMalloc(&h->d_draws, n * NDRAW * sizeof(double)));
  CK(cudaMalloc(&h->d_done, n));
  CK(cudaMemset(h->d_heading, 0, n * HEADING_SLOTS * sizeof(double)));
  CK(cudaMemset(h->d_draws, 0, n * NDRAW * sizeof(double)));
  CK(cudaMemset(h->d_done, 0, n));
  int rc = h->precision == TSG_PRECISION_F32 ? setup_model<P32>(h, model, prop.multiProcessorCount)
                                             : setup_model<P64>(h, model, prop.multiProcessorCount);
  if (rc) return rc;
  CK(cudaMalloc(&h->d_counter, 4 * sizeof(int)));
  CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  if (ec.use_obs_noise) {   // the noise-free observation always has a home; tsg_set_real_obs redirects it
    CK(cudaMalloc(&h->d_realobs_own, (size_t)n_envs * ec.obs_dim * sizeof(double)));
    CK(cudaMemset(h->d_realobs_own, 0, (size_t)n_envs * ec.obs_dim * sizeof(double)));
    h->real_obs = h->d_realobs_own;
  }
  if (n_pool) {
    CK(cudaMalloc(&h->d_pool_obs, (size_t)n_pool * ec.obs_dim * sizeof(double)));
    if (ec.use_obs_noise) CK(cudaMalloc(&h->d_pool_real_obs, (size_t)n_pool * ec.obs_dim * sizeof(double)));
    CK(cudaMalloc(&h->d_lists, (size_t)2 * n_pool * sizeof(int)));
    CK(cudaMalloc(&h->d_counts, 4 * sizeof(int)));
    CK(cudaMemset(h->d_counts, 0, 4 * sizeof(int)));
    CK(cudaMalloc(&h->d_need_sync, n_envs));
  }
  tsg_init_records_kernel<<<((int)n + 127) / 128, 128>>>(h->d_state, (int)n, h->d_qpos0);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return 0;
}

int tsg_create(const TsgModel* model, const TsgEnvConfig* cfg, int n_envs, int device, long long env_id_base,
               TsgHandle** out) {
  return tsg_create_opts(model, cfg, n_envs, 0, device, env_id_base, TSG_PRECISION_F64, out);
}
int tsg_create_pooled(const TsgModel* model, const TsgEnvConfig* cfg, int n_envs, int n_pool, int device,
                      long long env_id_base, TsgHandle** out) {
  return tsg_create_opts(model, cfg, n_envs, n_pool, device, env_id_base, TSG_PRECISION_F64, out);
}
int tsg_create_opts(const TsgModel* model, const TsgEnvConfig* cfg, int n_envs, int n_pool, int device,
                    long long env_id_base, int precision, TsgHandle** out) {
  if (!model || !cfg || !out) FAIL("tsg_create: null argument");
  if (n_envs < 1) FAIL("tsg_create: n_envs must be >= 1");
  if (n_pool < 0) FAIL("tsg_create: n_pool must be >= 0");
  if (precision != TSG_PRECISION_F64 && precision != TSG_PRECISION_F32) FAIL("tsg_create: bad precision");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); FAIL("tsg_create: no CUDA device (libtsg has no CPU path)"); }
  if (device < 0 || device >= ndev) FAIL("tsg_create: bad device index");
  CK(cudaSetDevice(device));
  TsgHandle* h = new TsgHandle();
  memset(h, 0, sizeof(*h));
  h->device = device; h->n_envs = n_envs; h->n_pool = n_pool; h->env_id_base = env_id_base; h->precision = precision;
  int rc = create_impl(h, model, cfg);
  if (rc) { std::string keep = g_err; tsg_destroy(h); g_err = keep; return rc; }   // no leak on a failed create
  *out = h;
  return 0;
}

int tsg_destroy(TsgHandle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  void* ptrs[] = {h->d_model, h->d_cfg, h->d_hdata, h->d_qpos0, h->d_state, h->d_heading, h->d_draws, h->d_done, h->d_ctrl,
                  h->d_obs, h->d_reward, h->d_info, h->d_termobs, h->d_tmp, h->d_mask, h->d_counter, h->d_spill, h->d_pool_obs,
                  h->d_pool_real_obs, h->d_lists, h->d_counts, h->d_need_sync, h->d_realobs_own, h->d_params, h->d_prange};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return 0;
}
int tsg_num_envs(const TsgHandle* h) { return h ? h->n_envs : -1; }
int tsg_obs_dim(const TsgHandle* h) { return h ? h->obs_dim : -1; }
int tsg_launches(const TsgHandle* h) { return h ? h->launches : -1; }
int tsg_precision(const TsgHandle* h) { return h ? h->precision : -1; }
int tsg_pool_stats_host(TsgHandle* h, int* counts3) {
  if (!h || !counts3) FAIL("tsg_pool_stats_host: null argument");
  counts3[0] = counts3[1] = counts3[2] = 0;
  if (!h->n_pool) return 0;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(counts3, h->d_counts, 3 * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}
int tsg_kernel_config(const TsgHandle* h, int* warps_per_cta, int* smem_bytes_out, int* regs_per_thread) {
  if (!h) FAIL("tsg_kernel_config: null handle");
  if (warps_per_cta) *warps_per_cta = (h->shape ? TB_WARPS_SMALL : TB_WARPS) * 100 + G;  // warps per CTA * 100 + lanes per env
  if (smem_bytes_out) *smem_bytes_out = (int)h->smem;
  if (regs_per_thread) *regs_per_thread = h->regs;
  return 0;
}

static StepIO base_io(TsgHandle* h) {
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.state = h->d_state; io.heading = h->d_heading; io.draws = h->d_draws;
  io.n_envs = h->n_envs; io.env_id_base = h->env_id_base;
  io.n_pool = h->n_pool; io.pool_obs = h->d_pool_obs; io.pool_real_obs = h->d_pool_real_obs;
  io.real_obs = h->real_obs;
  return io;
}

int tsg_reset(TsgHandle* h, const uint8_t* mask_dev, unsigned long long seed, const double* draws_in_dev,
              double* obs_dev, float* obs32_dev, double* term_obs_dev, void* stream) {
  if (!h) FAIL("tsg_reset: null handle");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  StepIO io = base_io(h);
  io.mask = mask_dev; io.seed = seed; io.obs = obs_dev; io.obs32 = obs32_dev; io.term_obs = term_obs_dev;
  if (draws_in_dev) {
    CK(cudaMemcpyAsync(h->d_draws, draws_in_dev, (size_t)h->n_envs * NDRAW * sizeof(double), cudaMemcpyDeviceToDevice, s));
    io.explicit_draws = 1;
  }
  if (zero_counters(h, s)) return -2;
  return launch_env<MODE_RESET>(h, io, s, 0);
}

int tsg_step(TsgHandle* h, const void* ctrl_dev, int ctrl_dtype, double* obs_dev, float* obs32_dev, double* reward_dev,
             uint8_t* done_dev, double* info_dev, int auto_reset, unsigned long long seed, double* term_obs_dev,
             void* stream) {
  if (!h) FAIL("tsg_step: null handle");
  if (!ctrl_dev) FAIL("tsg_step: ctrl_dev is null");
  if (ctrl_dtype != TSG_CTRL_F64 && ctrl_dtype != TSG_CTRL_F32) FAIL("tsg_step: bad ctrl_dtype");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  StepIO io = base_io(h);
  if (ctrl_dtype == TSG_CTRL_F64) io.ctrl64 = (const double*)ctrl_dev; else io.ctrl32 = (const float*)ctrl_dev;
  io.obs = obs_dev; io.obs32 = obs32_dev; io.reward = reward_dev; io.info = info_dev;
  io.done = done_dev ? done_dev : h->d_done;
  io.seed = seed;
  if (!auto_reset) io.n_pool = 0;  // the pool only advances on auto-resetting handles
  if (zero_counters(h, s)) return -2;   // one memset serves the step launch and the reset launch that may follow
  int rc = launch_env<MODE_STEP>(h, io, s, 0);
  if (rc) return rc;
  if (auto_reset) {
    const uint8_t* mask = io.done;
    if (h->n_pool) {  // hand pre-warmed slots to the done envs; only the remainder resets synchronously
      tsg_assign_kernel<<<1, 1024, 0, s>>>(h->d_state, h->d_heading, io.done, h->d_need_sync, obs_dev, obs32_dev, term_obs_dev,
                                           h->d_pool_obs, h->d_pool_real_obs, h->real_obs, h->d_lists, h->d_counts, h->n_envs,
                                           h->n_pool, h->obs_dim, h->ready_phase);
      CK(cudaGetLastError());
      h->launches++;
      if (h->per_env) {
        tsg_assign_params_kernel<<<h->n_pool < 1024 ? h->n_pool : 1024, 64, 0, s>>>(h->d_params, h->d_lists, h->d_counts, h->n_envs, h->n_pool);
        CK(cudaGetLastError());
        h->launches++;
      }
      mask = h->d_need_sync;
    }
    StepIO r = base_io(h);
    r.mask = mask; r.seed = seed; r.obs = obs_dev; r.obs32 = obs32_dev; r.term_obs = term_obs_dev;
    rc = launch_env<MODE_RESET>(h, r, s, 1);   // warps whose ten envs need no reset leave after one mask read
  }
  return rc;
}

int tsg_set_real_obs(TsgHandle* h, double* real_obs_dev) {
  if (!h) FAIL("tsg_set_real_obs: null handle");
  if (!h->d_realobs_own) FAIL("tsg_set_real_obs: the handle was created without use_obs_noise");
  h->real_obs = real_obs_dev ? real_obs_dev : h->d_realobs_own;
  return 0;
}
int tsg_get_real_obs_host(TsgHandle* h, double* real_obs) {
  if (!h || !real_obs) FAIL("tsg_get_real_obs_host: null argument");
  if (!h->real_obs) FAIL("tsg_get_real_obs_host: the handle was created without use_obs_noise");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(real_obs, h->real_obs, (size_t)h->n_envs * h->obs_dim * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

int tsg_forward(TsgHandle* h, double* obs_dev, double* info_dev, void* stream) {
  if (!h) FAIL("tsg_forward: null handle");
  CK(cudaSetDevice(h->device));
  StepIO io = base_io(h);
  io.obs = obs_dev; io.info = info_dev;
  if (zero_counters(h, (cudaStream_t)stream)) return -2;
  return launch_env<MODE_FORWARD>(h, io, (cudaStream_t)stream, 0);
}

// ---- per-env parameters
// first use: rows of every env and pool slot = the nominal row, and the handle switches to the per-env kernels
static int enable_params(TsgHandle* h) {
  if (h->per_env) return 0;
  size_t n = (size_t)h->n_envs + (size_t)h->n_pool;
  double pr[3 * NPARAM];
  for (int i = 0; i < NPARAM; i++) { pr[i] = h->nominal[i]; pr[NPARAM + i] = 1; pr[2 * NPARAM + i] = 1; }
  if (!h->d_prange) CK(cudaMalloc(&h->d_prange, sizeof(pr)));
  CK(cudaMalloc(&h->d_params, n * NPARAM * sizeof(double)));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(h->d_prange, pr, sizeof(pr), cudaMemcpyHostToDevice));
  tsg_fill_params_kernel<<<(int)((n * NPARAM + 255) / 256), 256>>>(h->d_params, (int)n, h->d_prange);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  int rc;
  if (h->precision == TSG_PRECISION_F32) rc = h->shape == 1 ? note_kernel<PerEnv<P32>, MODE_STEP, TB_WARPS_SMALL, TB_EPW_SMALL>(h) : note_kernel<PerEnv<P32>, MODE_STEP, TB_WARPS>(h);
  else rc = h->shape == 1 ? note_kernel<PerEnv<P64>, MODE_STEP, TB_WARPS_SMALL, TB_EPW_SMALL>(h) : note_kernel<PerEnv<P64>, MODE_STEP, TB_WARPS>(h);
  if (rc) return rc;
  h->per_env = 1;
  return 0;
}

int tsg_set_param_ranges(TsgHandle* h, const double* lo, const double* hi) {
  if (!h) FAIL("tsg_set_param_ranges: null handle");
  if (!lo != !hi) FAIL("tsg_set_param_ranges: lo and hi must both be given or both be NULL");
  CK(cudaSetDevice(h->device));
  if (!lo) {   // off: rows stay as they are at later resets
    if (h->per_env) { CK(cudaDeviceSynchronize()); h->ranges_on = 0; }
    return 0;
  }
  std::string err = check_param_ranges(lo, hi);
  if (!err.empty()) FAIL("tsg_set_param_ranges: " + err);
  int rc = enable_params(h);
  if (rc) return rc;
  CK(cudaDeviceSynchronize());   // no launch in flight reads the ranges being replaced
  CK(cudaMemcpy(h->d_prange + NPARAM, lo, NPARAM * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_prange + 2 * NPARAM, hi, NPARAM * sizeof(double), cudaMemcpyHostToDevice));
  h->ranges_on = 1;
  return 0;
}

int tsg_set_env_params(TsgHandle* h, const double* params_dev, const uint8_t* mask_dev, void* stream) {
  if (!h || !params_dev) FAIL("tsg_set_env_params: null argument");
  if (h->n_pool > 0)
    FAIL("tsg_set_env_params: the handle has a reset pool; an env that receives a pool slot takes the slot's row, "
         "which would replace an explicit row (create the handle with n_pool = 0)");
  CK(cudaSetDevice(h->device));
  int rc = enable_params(h);
  if (rc) return rc;
  size_t cnt = (size_t)h->n_envs * NPARAM;
  tsg_set_params_kernel<<<(int)((cnt + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_params, h->n_envs, params_dev, mask_dev);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

int tsg_get_env_params(TsgHandle* h, double* params_dev, void* stream) {
  if (!h || !params_dev) FAIL("tsg_get_env_params: null argument");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  size_t cnt = (size_t)h->n_envs * NPARAM;
  if (h->per_env) {
    CK(cudaMemcpyAsync(params_dev, h->d_params, cnt * sizeof(double), cudaMemcpyDeviceToDevice, s));
    return 0;
  }
  // without per-env parameters every env runs the nominal row; the nominal row comes from the host once
  if (!h->d_prange) {
    CK(cudaMalloc(&h->d_prange, 3 * NPARAM * sizeof(double)));
    CK(cudaMemcpy(h->d_prange, h->nominal, NPARAM * sizeof(double), cudaMemcpyHostToDevice));
  }
  tsg_fill_params_kernel<<<(int)((cnt + 255) / 256), 256, 0, s>>>(params_dev, h->n_envs, h->d_prange);
  CK(cudaGetLastError());
  h->launches++;
  return 0;
}

// ---- host-buffer helpers
static int ensure(double** p, size_t count) {
  if (*p) return 0;
  CK(cudaMalloc(p, count * sizeof(double)));
  return 0;
}
// mj_forward after a host-side state write, on the handle's own stream, synchronous (set_state of the single-env API)
int tsg_forward_host(TsgHandle* h, double* obs, double* info) {
  if (!h) FAIL("tsg_forward_host: null handle");
  CK(cudaSetDevice(h->device));
  size_t n = h->n_envs, od = h->obs_dim;
  if (ensure(&h->d_obs, n * od) || ensure(&h->d_info, n * INFO_DIM)) return -2;
  cudaStream_t s = h->own_stream;
  int rc = tsg_forward(h, h->d_obs, h->d_info, s);
  if (rc) return rc;
  if (obs) CK(cudaMemcpyAsync(obs, h->d_obs, n * od * 8, cudaMemcpyDeviceToHost, s));
  if (info) CK(cudaMemcpyAsync(info, h->d_info, n * INFO_DIM * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}
int tsg_get_state_host(TsgHandle* h, double* qpos, double* qvel, double* act, double* warm, double* ctrl) {
  if (!h) FAIL("tsg_get_state_host: null handle");
  CK(cudaSetDevice(h->device));
  size_t n = h->n_envs;
  if (ensure(&h->d_tmp, n * (NQ + 2 * NV + 2 * NACT))) return -2;
  double *dq = h->d_tmp, *dv = dq + n * NQ, *dw = dv + n * NV, *dc = dw + n * NV, *da = dc + n * NACT;
  CK(cudaDeviceSynchronize());
  tsg_gather_kernel<<<(h->n_envs + 127) / 128, 128>>>(h->d_state, h->n_envs, dq, dv, da, dw, dc);
  CK(cudaGetLastError());
  if (qpos) CK(cudaMemcpy(qpos, dq, n * NQ * 8, cudaMemcpyDeviceToHost));
  if (qvel) CK(cudaMemcpy(qvel, dv, n * NV * 8, cudaMemcpyDeviceToHost));
  if (warm) CK(cudaMemcpy(warm, dw, n * NV * 8, cudaMemcpyDeviceToHost));
  if (ctrl) CK(cudaMemcpy(ctrl, dc, n * NACT * 8, cudaMemcpyDeviceToHost));
  if (act) CK(cudaMemcpy(act, da, n * NACT * 8, cudaMemcpyDeviceToHost));
  return 0;
}
int tsg_set_state_host(TsgHandle* h, const double* qpos, const double* qvel, const double* act, const double* warm,
                       const double* ctrl) {
  if (!h) FAIL("tsg_set_state_host: null handle");
  CK(cudaSetDevice(h->device));
  size_t n = h->n_envs;
  if (ensure(&h->d_tmp, n * (NQ + 2 * NV + 2 * NACT))) return -2;
  double *dq = h->d_tmp, *dv = dq + n * NQ, *dw = dv + n * NV, *dc = dw + n * NV, *da = dc + n * NACT;
  CK(cudaDeviceSynchronize());
  if (qpos) CK(cudaMemcpy(dq, qpos, n * NQ * 8, cudaMemcpyHostToDevice));
  if (qvel) CK(cudaMemcpy(dv, qvel, n * NV * 8, cudaMemcpyHostToDevice));
  if (warm) CK(cudaMemcpy(dw, warm, n * NV * 8, cudaMemcpyHostToDevice));
  if (ctrl) CK(cudaMemcpy(dc, ctrl, n * NACT * 8, cudaMemcpyHostToDevice));
  if (act) CK(cudaMemcpy(da, act, n * NACT * 8, cudaMemcpyHostToDevice));
  tsg_scatter_kernel<<<(h->n_envs + 127) / 128, 128>>>(h->d_state, h->n_envs, qpos ? dq : nullptr, qvel ? dv : nullptr,
                                                        act ? da : nullptr, warm ? dw : nullptr, ctrl ? dc : nullptr);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return 0;
}
int tsg_get_records_host(TsgHandle* h, double* records) {
  if (!h || !records) FAIL("tsg_get_records_host: null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(records, h->d_state, (size_t)h->n_envs * STATE_STRIDE * 8, cudaMemcpyDeviceToHost));
  return 0;
}
int tsg_set_records_host(TsgHandle* h, const double* records) {
  if (!h || !records) FAIL("tsg_set_records_host: null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(h->d_state, records, (size_t)h->n_envs * STATE_STRIDE * 8, cudaMemcpyHostToDevice));
  return 0;
}
// the heading rings the records' cursors (head_n / head_pos) point into: part of an env-state checkpoint
int tsg_get_heading_host(TsgHandle* h, double* heading) {
  if (!h || !heading) FAIL("tsg_get_heading_host: null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(heading, h->d_heading, (size_t)h->n_envs * HEADING_SLOTS * 8, cudaMemcpyDeviceToHost));
  return 0;
}
int tsg_set_heading_host(TsgHandle* h, const double* heading) {
  if (!h || !heading) FAIL("tsg_set_heading_host: null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(h->d_heading, heading, (size_t)h->n_envs * HEADING_SLOTS * 8, cudaMemcpyHostToDevice));
  return 0;
}
int tsg_get_draws_host(TsgHandle* h, double* draws) {
  if (!h || !draws) FAIL("tsg_get_draws_host: null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(draws, h->d_draws, (size_t)h->n_envs * NDRAW * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int tsg_step_host(TsgHandle* h, const double* ctrl, double* obs, double* reward, uint8_t* done, double* info,
                  int auto_reset, unsigned long long seed, double* term_obs) {
  if (!h || !ctrl) FAIL("tsg_step_host: null argument");
  CK(cudaSetDevice(h->device));
  size_t n = h->n_envs, od = h->obs_dim;
  if (ensure(&h->d_ctrl, n * NACT) || ensure(&h->d_obs, n * od) || ensure(&h->d_reward, n) ||
      ensure(&h->d_info, n * INFO_DIM) || ensure(&h->d_termobs, n * od)) return -2;
  cudaStream_t s = h->own_stream;
  CK(cudaMemcpyAsync(h->d_ctrl, ctrl, n * NACT * 8, cudaMemcpyHostToDevice, s));
  int rc = tsg_step(h, h->d_ctrl, TSG_CTRL_F64, h->d_obs, nullptr, h->d_reward, h->d_done, info ? h->d_info : nullptr,
                    auto_reset, seed, term_obs ? h->d_termobs : nullptr, s);
  if (rc) return rc;
  if (obs) CK(cudaMemcpyAsync(obs, h->d_obs, n * od * 8, cudaMemcpyDeviceToHost, s));
  if (reward) CK(cudaMemcpyAsync(reward, h->d_reward, n * 8, cudaMemcpyDeviceToHost, s));
  if (done) CK(cudaMemcpyAsync(done, h->d_done, n, cudaMemcpyDeviceToHost, s));
  if (info) CK(cudaMemcpyAsync(info, h->d_info, n * INFO_DIM * 8, cudaMemcpyDeviceToHost, s));
  if (term_obs) CK(cudaMemcpyAsync(term_obs, h->d_termobs, n * od * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}
int tsg_reset_host(TsgHandle* h, const uint8_t* mask, unsigned long long seed, const double* draws_in, double* obs) {
  if (!h) FAIL("tsg_reset_host: null handle");
  CK(cudaSetDevice(h->device));
  size_t n = h->n_envs, od = h->obs_dim;
  if (ensure(&h->d_obs, n * od)) return -2;
  cudaStream_t s = h->own_stream;
  if (mask) {
    if (!h->d_mask) CK(cudaMalloc(&h->d_mask, n));
    CK(cudaMemcpyAsync(h->d_mask, mask, n, cudaMemcpyHostToDevice, s));
  }
  double* d_draws_in = nullptr;
  if (draws_in) {
    if (ensure(&h->d_tmp, n * (NQ + 2 * NV + 2 * NACT))) return -2;
    d_draws_in = h->d_tmp;
    CK(cudaMemcpyAsync(d_draws_in, draws_in, n * NDRAW * 8, cudaMemcpyHostToDevice, s));
  }
  int rc = tsg_reset(h, mask ? h->d_mask : nullptr, seed, d_draws_in, h->d_obs, nullptr, nullptr, s);
  if (rc) return rc;
  if (obs) CK(cudaMemcpyAsync(obs, h->d_obs, n * od * 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}
